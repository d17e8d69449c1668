/*
 * dcmt.h -- C ABI of libdcmt.so: the B200 (sm_100a) replacement for the depth-completion hot path of
 * PatrizioPerugini/depth_completion_MT.
 *
 * The reference has no FFI layer: its hot path is three groups of free C++ functions on cv::Mat
 *   (a1) img_completion                    src/DC_lidar_only/img_completion.cpp:17-20
 *   (a2) interpolate_with_superpixels      src/DC_lidar_camera/img_completion_lc.cpp:34-38
 *   (a4-a9) calculateMeasuementDerivatives / get_initial_disparity / optimize_IG /
 *           retrieve_optimized_depth / final GaussianBlur
 *                                          src/DC_stereo_lidar/main_sl.cpp:715,747,804,846,863,1253
 * Each entry point below names the reference function it replaces.  include/img_completion.h is
 * the C++ shim that keeps the reference's own signatures on top of this ABI.
 *
 * Conventions
 *   - plain pointers and sizes only; no C++/torch/OpenCV types cross this boundary;
 *   - every function returns DCMT_OK (0) or a negative DCMT_E_* code, never throws, never prints;
 *     dcmt_last_error() returns a thread-local description of the last failure;
 *   - un-suffixed entry points take DEVICE pointers, enqueue all work on `cuda_stream`
 *     (a cudaStream_t passed as void*, NULL = legacy default stream) and return without
 *     synchronising; `*_host` variants take HOST pointers, copy in/out and synchronise;
 *   - images are row-major float32 (CV_32FC1), `pitch_bytes` between rows (0 = cols*4),
 *     `frame_stride_bytes` between consecutive frames of a batch (0 = rows*pitch);
 *   - input and output must not alias; the library keeps a cached per-(device,stream) workspace,
 *     nothing else is retained after return;
 *   - threading: dcmt_last_error() is thread-local.  Un-suffixed (device-pointer) entry points may be called from
 *     several threads as long as calls that share a (device, stream) pair are ordered by the caller, as CUDA itself
 *     requires (the workspace and the read-back buffer of DCMT_PATH_AUTO are cached per pair).  `*_host` entry points
 *     share three internal streams per device and take a per-device mutex for the duration of the call: threads on
 *     different devices run concurrently, threads on the same device take turns.  On every return path, including
 *     errors, a `*_host` call has drained its streams: no copy into the caller's buffers is in flight afterwards;
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails with
 *     DCMT_E_CUDA.
 */
#ifndef DCMT_H_
#define DCMT_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define DCMT_API
#else
#define DCMT_API __attribute__((visibility("default")))
#endif

#define DCMT_VERSION 200 /* 0.2.0 */

enum {
    DCMT_OK = 0,
    DCMT_E_BADARG = -1,      /* null pointer, non-positive size, bad pitch, aliasing in/out */
    DCMT_E_UNSUPPORTED = -2, /* valid request this build cannot serve */
    DCMT_E_CUDA = -3,        /* CUDA runtime error (see dcmt_last_error) */
    DCMT_E_NOMEM = -4        /* workspace allocation failed */
};

/* blur_type of img_completion (img_completion.cpp:172-189): any string other than "gaussian" /
 * "bilateral" means no blur. */
enum { DCMT_BLUR_NONE = 0, DCMT_BLUR_GAUSSIAN = 1, DCMT_BLUR_BILATERAL = 2 };

/* kernel path selection (flags argument) */
enum {
    /* fused strict-q8 kernels with in-kernel validation; frames that turn out not to be strict q8 (any pixel that is
     * neither 0 nor k/256 with 26 <= k <= 25574) are redone by the generic pipeline.  Always correct; reads one
     * int32 per frame back at the end of the call, i.e. synchronises the stream once. */
    DCMT_PATH_AUTO = 0,
    /* generic float32 multi-kernel pipeline: any finite input, fully asynchronous */
    DCMT_PATH_GENERIC = 1,
    /* fused kernels without validation, fully asynchronous (CUDA-graph capturable): the CALLER guarantees strict q8
     * input (e.g. KITTI uint16 PNG / 256, main.cpp:75-82); other input gives undefined output.  Shapes / blur
     * types the fused kernels do not serve (bilateral, frames under 32x32) still use the generic pipeline. */
    DCMT_PATH_FUSED = 2,
    /* float32 frames that are NOT strict q8 -- e.g. the cv::normalize'd depth the stereo program completes
     * (main_sl.cpp:522-540) -- on the same fused kernels: the inverted values of a frame's valid pixels are sorted into a
     * per-frame dictionary and replaced by their ranks (every stage between the inversion and the blur only selects among
     * its inputs, so any monotone code gives the same selections), and the tail decodes before the float32 Gaussian.
     * Bit-identical to the reference with blur none, within 1e-4 with the Gaussian.  Frames with more than 32768 valid
     * pixels or a NaN are redone by the generic pipeline (one read-back, like DCMT_PATH_AUTO).  DCMT_PATH_AUTO tries the
     * strict-q8 kernels first, then this, then the generic pipeline. */
    DCMT_PATH_RANK = 3
};

/* per-frame statistics, DCMT_STATS_STRIDE int32 per frame (device memory for the async entry
 * points, host memory for *_host), all optional (NULL):
 *   [0] passes the reference's `while` loop executes (img_completion.cpp:146-166), >= 1
 *   [1] holes counted by the first loop pass (= holes left after the first 31x31 fill)
 *   [2] holes counted by the first 31x31 fill (= holes left after column extrapolation)
 *   [3] path that produced the frame: 0 generic, 1 fused strict-q8, 2 fused through the float32 dictionary (DCMT_PATH_RANK) */
#define DCMT_STATS_STRIDE 4

DCMT_API int dcmt_version(void);
/* "cuda sm_100a" for the product library; the test-only CPU emulator build of the same sources says so here, and the
 * Python package refuses to load anything that does not start with "cuda" */
DCMT_API const char *dcmt_build_info(void);
DCMT_API const char *dcmt_last_error(void);
DCMT_API const char *dcmt_status_string(int status);
/* number of visible CUDA devices, or a negative DCMT_E_CUDA */
DCMT_API int dcmt_device_count(void);
/* frees every cached workspace of the calling process (all devices) */
DCMT_API int dcmt_release_workspaces(void);
/* number of CUDA kernels this library has launched in the calling process (monotonic; bench.py reports the
 * difference across its timed region as `gpu_launches`) */
DCMT_API long long dcmt_launch_count(void);
/* per-kernel timing of the fused path: between begin and end every chunk's k_q8_front (with its two set-up kernels)
 * and k_q8_tail (with fix-up and stats kernels) are bracketed by CUDA events on the launch stream; end waits for
 * them and returns the summed milliseconds and the number of chunks.  Not thread-safe with concurrent callers. */
DCMT_API int dcmt_profile_begin(void);
DCMT_API int dcmt_profile_end(double *front_ms, double *tail_ms, long long *chunks);
/* page-locked host buffers for the *_host entry points (their copies are asynchronous and overlap the kernels only
 * for page-locked memory).  write_combined != 0: for INPUT buffers the host only writes sequentially (faster for the
 * device to read, very slow for the host to read back). */
DCMT_API int dcmt_host_alloc(size_t bytes, int write_combined, void **out);
DCMT_API int dcmt_host_free(void *p);
/* bytes of device workspace the library caches for a call of this shape */
DCMT_API size_t dcmt_workspace_bytes(int rows, int cols, int n_frames);

/* (a1) replaces img_completion(const cv::Mat&, cv::Mat&, const bool& extr, const std::string&)
 * -- src/DC_lidar_only/img_completion.cpp:17-204.  `extr` is ignored by the reference (:103) and
 * has no counterpart here. */
DCMT_API int dcmt_img_completion_f32(const float *sparse, float *dense, int rows, int cols, size_t pitch_bytes,
                                     size_t frame_stride_bytes, int n_frames, int blur_type, int flags,
                                     int32_t *stats_or_null, void *cuda_stream);
DCMT_API int dcmt_img_completion_f32_host(const float *sparse, float *dense, int rows, int cols, size_t pitch_bytes,
                                          size_t frame_stride_bytes, int n_frames, int blur_type, int flags,
                                          int32_t *stats_or_null);

/* (a1, KITTI on-disk format) replaces the caller's sequence main.cpp:75-93: the uint16 payload of a KITTI depth PNG
 * (cv::imread(..., IMREAD_ANYDEPTH)), convertTo(CV_32F, 1.0 / 256.0) (main.cpp:79) and img_completion (:93) in one
 * call.  Input pixels are uint16 = metres * 256 (0 = empty), output is float32 metres as above.  Input and output have
 * their own pitches / frame strides in bytes (0 = dense).  uint16 input is strict q8 by construction, so the fused
 * kernels serve it without validation and the call never synchronises (DCMT_PATH_AUTO == DCMT_PATH_FUSED here);
 * it moves 6 instead of 8 bytes per pixel through HBM and halves the host-to-device copy of the *_host variant. */
DCMT_API int dcmt_img_completion_u16(const uint16_t *sparse_u16, float *dense, int rows, int cols, size_t in_pitch_bytes,
                                     size_t in_frame_stride_bytes, size_t out_pitch_bytes, size_t out_frame_stride_bytes,
                                     int n_frames, int blur_type, int flags, int32_t *stats_or_null, void *cuda_stream);
DCMT_API int dcmt_img_completion_u16_host(const uint16_t *sparse_u16, float *dense, int rows, int cols,
                                          size_t in_pitch_bytes, size_t in_frame_stride_bytes, size_t out_pitch_bytes,
                                          size_t out_frame_stride_bytes, int n_frames, int blur_type, int flags,
                                          int32_t *stats_or_null);

/* (a1, KITTI on-disk format in and out) the same with the output in KITTI's format as well: uint16 = metres * 256, 0 = empty
 * -- what a caller that stores the completed map gets from convertTo(CV_16U, 256) in front of cv::imwrite, i.e. the rule of
 * dcmt_depth_to_u16 applied to the float32 output of dcmt_img_completion_u16.  On the fused kernels the tail stores the
 * uint16 values directly (the float32 output is an integer multiple of 2^-16 m there); with blur none the result is
 * lossless (u / 256 equals the float32 output).  Frames the fused kernels do not serve (bilateral, frames under 32x32,
 * DCMT_PATH_GENERIC) are completed in float32 and converted.  Pitches / frame strides in bytes (0 = dense), flags, stats
 * and the never-synchronising behaviour as for dcmt_img_completion_u16; the host-to-device and device-to-host copies
 * of the *_host variants both move 2 bytes per pixel. */
DCMT_API int dcmt_img_completion_u16_u16(const uint16_t *sparse_u16, uint16_t *dense_u16, int rows, int cols, size_t in_pitch_bytes,
                                         size_t in_frame_stride_bytes, size_t out_pitch_bytes, size_t out_frame_stride_bytes,
                                         int n_frames, int blur_type, int flags, int32_t *stats_or_null, void *cuda_stream);
DCMT_API int dcmt_img_completion_u16_u16_host(const uint16_t *sparse_u16, uint16_t *dense_u16, int rows, int cols,
                                              size_t in_pitch_bytes, size_t in_frame_stride_bytes, size_t out_pitch_bytes,
                                              size_t out_frame_stride_bytes, int n_frames, int blur_type, int flags,
                                              int32_t *stats_or_null);

/* cv::Mat::convertTo(CV_16U, 256.0) of float32 depth maps (device pointers): u = saturate_cast<uint16_t>(cvRound(v * 256)) --
 * the product is exact, rounding is half to even, the result is clamped to [0, 65535] and NaN gives 0.  (OpenCV's x86
 * build gives 0 instead of 65535 where v * 256 is +inf or at least 2^31, because its cvRound overflows there; depth
 * maps never get near that.)  For float-output callers -- the dictionary path, the stereo chain -- that store KITTI
 * PNGs.  Pitches / frame strides in bytes (0 = dense); overlapping input and output ranges are DCMT_E_BADARG. */
DCMT_API int dcmt_depth_to_u16(const float *depth, uint16_t *out, int rows, int cols, size_t in_pitch_bytes,
                               size_t in_frame_stride_bytes, size_t out_pitch_bytes, size_t out_frame_stride_bytes, int n_frames,
                               void *cuda_stream);

/* (e) the host-pointer entry points over several GPUs of one box: north_star's "batches are partitioned frame-wise
 * across the 8 B200s" for a C++ caller of the library (one process, one thread).  The frames of the call are split into
 * one contiguous block per device; chunks of the blocks flow H2D -> kernels -> D2H on three streams per device, all
 * enqueued by the calling thread; there is no exchange between devices.  `devices` lists CUDA device ordinals
 * (n_devices >= 1, no repeats); devices == NULL uses the first n_devices visible devices, or all of them when
 * n_devices <= 0.  Page-locked host buffers (dcmt_host_alloc) are needed for the copies to overlap.  The caller's
 * current device is restored on return.  Results are identical to the single-device call. */
DCMT_API int dcmt_img_completion_f32_host_multi(const float *sparse, float *dense, int rows, int cols, size_t pitch_bytes,
                                                size_t frame_stride_bytes, int n_frames, int blur_type, int flags,
                                                int32_t *stats_or_null, const int *devices_or_null, int n_devices);
DCMT_API int dcmt_img_completion_u16_host_multi(const uint16_t *sparse_u16, float *dense, int rows, int cols,
                                                size_t in_pitch_bytes, size_t in_frame_stride_bytes, size_t out_pitch_bytes,
                                                size_t out_frame_stride_bytes, int n_frames, int blur_type, int flags,
                                                int32_t *stats_or_null, const int *devices_or_null, int n_devices);
DCMT_API int dcmt_img_completion_u16_u16_host_multi(const uint16_t *sparse_u16, uint16_t *dense_u16, int rows, int cols,
                                                    size_t in_pitch_bytes, size_t in_frame_stride_bytes, size_t out_pitch_bytes,
                                                    size_t out_frame_stride_bytes, int n_frames, int blur_type, int flags,
                                                    int32_t *stats_or_null, const int *devices_or_null, int n_devices);
DCMT_API int dcmt_interpolate_with_superpixels_f32_host_multi(const float *sparse, const int32_t *labels, int n_clusters,
                                                              float *dense, int rows, int cols, size_t pitch_bytes,
                                                              size_t frame_stride_bytes, int n_frames, int use_superpixel,
                                                              int flags, int32_t *stats_or_null, const int *devices_or_null,
                                                              int n_devices);
/* measurement aid: the host pipeline of the calls above with the kernels left out -- the same buffers, chunking and
 * streams; the float32 variant echoes the input to the output, the uint16 variant returns zeros.  Its rate is the
 * ceiling the host <-> device links put on the end-to-end rate (bench.py: e2e.copy_ceiling).  devices == NULL and
 * n_devices == 0: the current device. */
DCMT_API int dcmt_debug_host_copy_f32(const float *in, float *out, int rows, int cols, int n_frames,
                                      const int *devices_or_null, int n_devices);
DCMT_API int dcmt_debug_host_copy_u16(const uint16_t *in, float *out, int rows, int cols, int n_frames,
                                      const int *devices_or_null, int n_devices);
/* the uint16-in, uint16-out pipeline (dcmt_img_completion_u16_u16_host); echoes the input to the output */
DCMT_API int dcmt_debug_host_copy_u16_u16(const uint16_t *in, uint16_t *out, int rows, int cols, int n_frames,
                                          const int *devices_or_null, int n_devices);

/* (a2) replaces interpolate_with_superpixels(Slic&, const cv::Mat&, cv::Mat&, const std::string&, int)
 * -- src/DC_lidar_camera/img_completion_lc.cpp:34-203.  `labels` is the Slic::clusters label map as
 * row-major int32 [row][col] (the reference stores [col][row], :83; the C++ shim transposes),
 * `n_clusters` = slic.centers.size(); labels outside [0, n_clusters) are never selected.  The
 * reference ignores blur_type here (Gaussian is unconditional, :183-192). */
DCMT_API int dcmt_interpolate_with_superpixels_f32(const float *sparse, const int32_t *labels, int n_clusters,
                                                   float *dense, int rows, int cols, size_t pitch_bytes,
                                                   size_t frame_stride_bytes, int n_frames, int use_superpixel,
                                                   int32_t *stats_or_null, void *cuda_stream);
DCMT_API int dcmt_interpolate_with_superpixels_f32_host(const float *sparse, const int32_t *labels, int n_clusters,
                                                        float *dense, int rows, int cols, size_t pitch_bytes,
                                                        size_t frame_stride_bytes, int n_frames, int use_superpixel,
                                                        int32_t *stats_or_null);

/* the same with an explicit kernel path (`flags` as for dcmt_img_completion_f32).  The plain entry points above use
 * DCMT_PATH_AUTO: strict-q8 frames (KITTI depth) run the fused guided front + fused tail, other frames the generic
 * float pipeline; the fused guided front needs n_clusters <= 65535. */
DCMT_API int dcmt_interpolate_with_superpixels_ex_f32(const float *sparse, const int32_t *labels, int n_clusters,
                                                      float *dense, int rows, int cols, size_t pitch_bytes,
                                                      size_t frame_stride_bytes, int n_frames, int use_superpixel,
                                                      int flags, int32_t *stats_or_null, void *cuda_stream);
DCMT_API int dcmt_interpolate_with_superpixels_ex_f32_host(const float *sparse, const int32_t *labels, int n_clusters,
                                                           float *dense, int rows, int cols, size_t pitch_bytes,
                                                           size_t frame_stride_bytes, int n_frames, int use_superpixel,
                                                           int flags, int32_t *stats_or_null);

/* (a2, KITTI on-disk format) main_lc.cpp:159-180 + :220 in one call: the uint16 payload of the KITTI depth PNG, its
 * convertTo(CV_32F, 1/256) and interpolate_with_superpixels.  Labels, n_clusters and use_superpixel as for
 * dcmt_interpolate_with_superpixels_f32; pitches / frame strides in bytes (0 = dense); flags and stats as for
 * dcmt_img_completion_u16 (uint16 input is strict q8: the fused guided front reads it directly unless n_clusters > 65535 or
 * DCMT_PATH_GENERIC, and the call never synchronises).  The output equals dcmt_interpolate_with_superpixels_ex_f32 on
 * sparse_u16 / 256; the _u16_u16 variants store it as KITTI uint16 by the rule of dcmt_depth_to_u16. */
DCMT_API int dcmt_interpolate_with_superpixels_u16(const uint16_t *sparse_u16, const int32_t *labels, int n_clusters, float *dense,
                                                   int rows, int cols, size_t in_pitch_bytes, size_t in_frame_stride_bytes,
                                                   size_t out_pitch_bytes, size_t out_frame_stride_bytes, int n_frames,
                                                   int use_superpixel, int flags, int32_t *stats_or_null, void *cuda_stream);
DCMT_API int dcmt_interpolate_with_superpixels_u16_host(const uint16_t *sparse_u16, const int32_t *labels, int n_clusters,
                                                        float *dense, int rows, int cols, size_t in_pitch_bytes,
                                                        size_t in_frame_stride_bytes, size_t out_pitch_bytes,
                                                        size_t out_frame_stride_bytes, int n_frames, int use_superpixel, int flags,
                                                        int32_t *stats_or_null);
DCMT_API int dcmt_interpolate_with_superpixels_u16_host_multi(const uint16_t *sparse_u16, const int32_t *labels, int n_clusters,
                                                              float *dense, int rows, int cols, size_t in_pitch_bytes,
                                                              size_t in_frame_stride_bytes, size_t out_pitch_bytes,
                                                              size_t out_frame_stride_bytes, int n_frames, int use_superpixel,
                                                              int flags, int32_t *stats_or_null, const int *devices_or_null,
                                                              int n_devices);
DCMT_API int dcmt_interpolate_with_superpixels_u16_u16(const uint16_t *sparse_u16, const int32_t *labels, int n_clusters,
                                                       uint16_t *dense_u16, int rows, int cols, size_t in_pitch_bytes,
                                                       size_t in_frame_stride_bytes, size_t out_pitch_bytes,
                                                       size_t out_frame_stride_bytes, int n_frames, int use_superpixel, int flags,
                                                       int32_t *stats_or_null, void *cuda_stream);
DCMT_API int dcmt_interpolate_with_superpixels_u16_u16_host(const uint16_t *sparse_u16, const int32_t *labels, int n_clusters,
                                                            uint16_t *dense_u16, int rows, int cols, size_t in_pitch_bytes,
                                                            size_t in_frame_stride_bytes, size_t out_pitch_bytes,
                                                            size_t out_frame_stride_bytes, int n_frames, int use_superpixel,
                                                            int flags, int32_t *stats_or_null);
DCMT_API int dcmt_interpolate_with_superpixels_u16_u16_host_multi(const uint16_t *sparse_u16, const int32_t *labels, int n_clusters,
                                                                  uint16_t *dense_u16, int rows, int cols, size_t in_pitch_bytes,
                                                                  size_t in_frame_stride_bytes, size_t out_pitch_bytes,
                                                                  size_t out_frame_stride_bytes, int n_frames, int use_superpixel,
                                                                  int flags, int32_t *stats_or_null, const int *devices_or_null,
                                                                  int n_devices);

/* parameters of the stereo refinement; dcmt_stereo_params_default() fills the values hard-coded in
 * main_sl.cpp, dcmt_stereo_params_official() those of main_sl_OFFICIAL.cpp:832-918. */
typedef struct dcmt_stereo_params {
    float baseline;         /* 0.54        main_sl.cpp:848,866 */
    float focal;            /* 959.791     main_sl.cpp:849,867 */
    float damp_factor;      /* 500   (OFFICIAL 1370)   :808 */
    float err_clip;         /* 255   (OFFICIAL 221)    :820-825 */
    float depth_clip;       /* 100   (OFFICIAL 80)     :875 */
    int32_t num_iterations; /* 4                       :805 */
    int32_t final_gauss;    /* 1     (OFFICIAL 0)      :1253 */
} dcmt_stereo_params;
DCMT_API void dcmt_stereo_params_default(dcmt_stereo_params *p);
DCMT_API void dcmt_stereo_params_official(dcmt_stereo_params *p, int num_iterations);

/* (a3-a9) replaces the sequence main_sl.cpp:1165-1253: EntryType fill from the two gray images,
 * calculateMeasuementDerivatives (:715), get_initial_disparity (:846), optimize_IG (:804, with
 * calculateObservationDerivatives :747 inlined), retrieve_optimized_depth (:863), GaussianBlur (:1253).
 * gray planes are uint8 row-major with pitch = cols; depth planes float32 with pitch = cols*4.
 * disp_out_or_null receives the refined disparity (the reference's disparity_IG after :1240). */
DCMT_API int dcmt_stereo_refine_f32(const float *depth_ig, const uint8_t *left_gray, const uint8_t *right_gray,
                                    float *depth_out, float *disp_out_or_null, int rows, int cols, int n_frames,
                                    const dcmt_stereo_params *params, void *cuda_stream);
DCMT_API int dcmt_stereo_refine_f32_host(const float *depth_ig, const uint8_t *left_gray, const uint8_t *right_gray,
                                         float *depth_out, float *disp_out_or_null, int rows, int cols, int n_frames,
                                         const dcmt_stereo_params *params);

/* the individual stereo functions, for callers that use them one by one (device pointers) */
/* (a4) calculateMeasuementDerivatives, main_sl.cpp:715-745: value plane -> dx, dy planes */
DCMT_API int dcmt_measurement_derivatives_f32(const float *value, float *dx, float *dy, int rows, int cols,
                                              int n_frames, void *cuda_stream);
/* (a5) get_initial_disparity, main_sl.cpp:846-861 (output pre-zeroed as at :1191) */
DCMT_API int dcmt_get_initial_disparity_f32(const float *depth, float *disp, int rows, int cols, int n_frames,
                                            float baseline, float focal, void *cuda_stream);
/* (a6+a7) optimize_IG, main_sl.cpp:804-843: value planes of both images, disparity in place */
DCMT_API int dcmt_optimize_ig_f32(const float *value_left, const float *value_right, float *disp, int rows, int cols,
                                  int n_frames, int num_iterations, float damp_factor, float err_clip,
                                  void *cuda_stream);
/* (a8) retrieve_optimized_depth, main_sl.cpp:863-885 (output pre-zeroed as at :1244) */
DCMT_API int dcmt_retrieve_optimized_depth_f32(const float *disp, float *depth, int rows, int cols, int n_frames,
                                               float baseline, float focal, float depth_clip, void *cuda_stream);

/* cv::cvtColor(COLOR_BGR2GRAY) on CV_8UC3 images (main_sl.cpp:1167,1171), the step in front of the EntryType fill:
 * OpenCV's 8-bit path is fixed point, gray = (3735 B + 19235 G + 9798 R + 16384) >> 15 -- bit-equal to OpenCV 4.13.
 * n_frames images follow each other at rows * pitch; pitches in bytes (0 = dense: cols * 3 / cols). */
DCMT_API int dcmt_bgr2gray_u8(const uint8_t *bgr, uint8_t *gray, int rows, int cols, size_t bgr_pitch_bytes,
                              size_t gray_pitch_bytes, int n_frames, void *cuda_stream);
DCMT_API int dcmt_bgr2gray_u8_host(const uint8_t *bgr, uint8_t *gray, int rows, int cols, size_t bgr_pitch_bytes,
                                   size_t gray_pitch_bytes, int n_frames);

/* cv::cvtColor(img, lab, COLOR_BGR2Lab) on CV_8UC3 images, the conversion in front of Slic::generate_superpixels
 * (main_lc.cpp:182-183; main_sl.cpp:438 in withSuperPixels): OpenCV's 8-bit path -- sRGB gamma and the Lab cube root by
 * table, XYZ and L, a, b in fixed point -- bit-equal to OpenCV 4.13 for all 2^24 colours.  CV_8UC3 Lab out (L * 255 / 100,
 * a + 128, b + 128).  n_frames images follow each other at rows * pitch; pitches in bytes (0 = dense: cols * 3).
 * Input and output byte ranges that overlap are DCMT_E_BADARG. */
DCMT_API int dcmt_bgr2lab_u8(const uint8_t *bgr, uint8_t *lab, int rows, int cols, size_t bgr_pitch_bytes,
                             size_t lab_pitch_bytes, int n_frames, void *cuda_stream);
DCMT_API int dcmt_bgr2lab_u8_host(const uint8_t *bgr, uint8_t *lab, int rows, int cols, size_t bgr_pitch_bytes,
                                  size_t lab_pitch_bytes, int n_frames);

/* (a3) the same four functions on the reference's OWN containers, so that its call sites (main_sl.cpp:1192-1246) need no
 * change of data layout:
 *   - EntryType matrices (main_sl.cpp:23-26: struct { float value; Eigen::Vector2f derivative; }, 12 bytes) as
 *     cv::Mat(rows, cols, CV_32FC(sizeof(EntryType))) (:1165,:1169): element (r, c) lives at
 *     data + r * row_step_bytes + c * elem_stride_bytes with elem_stride_bytes = 12 and row_step_bytes = Mat::step
 *     (= cols * 48 there: at<EntryType>() packs the 12-byte entries at the start of rows four times too wide);
 *   - CV_32FC1 matrices with a pitch, written IN PLACE the way the reference loops do: get_initial_disparity only
 *     writes where depth > 0 (:852), retrieve_optimized_depth only where disparity > 0 (:871); other pixels keep
 *     what the output held;
 *   - calculateMeasuementDerivatives writes derivative (x, y) of the interior entries and leaves the one-pixel border
 *     as the caller initialised it (:717-721); optimize_IG reads value and the STORED derivative.x() of the right
 *     matrix (:747-801) and value of the left one, and updates the disparity in place; reads at column index == cols
 *     (undefined in the reference) are 0.
 * Device-pointer variants enqueue on `cuda_stream`; `*_host` variants copy the used part of the rows in and the
 * modified data back.  rows <= 65535. */
DCMT_API int dcmt_entries_measurement_derivatives(void *entries, int rows, int cols, size_t row_step_bytes,
                                                  size_t elem_stride_bytes, void *cuda_stream);
DCMT_API int dcmt_entries_measurement_derivatives_host(void *entries, int rows, int cols, size_t row_step_bytes,
                                                       size_t elem_stride_bytes);
DCMT_API int dcmt_entries_optimize_ig(const void *entries_left, size_t left_row_step_bytes, const void *entries_right,
                                      size_t right_row_step_bytes, size_t elem_stride_bytes, float *disp,
                                      size_t disp_pitch_bytes, int rows, int cols, int num_iterations, float damp_factor,
                                      float err_clip, void *cuda_stream);
DCMT_API int dcmt_entries_optimize_ig_host(const void *entries_left, size_t left_row_step_bytes, const void *entries_right,
                                           size_t right_row_step_bytes, size_t elem_stride_bytes, float *disp,
                                           size_t disp_pitch_bytes, int rows, int cols, int num_iterations,
                                           float damp_factor, float err_clip);
DCMT_API int dcmt_get_initial_disparity_mat_f32(const float *depth, size_t depth_pitch_bytes, float *disp,
                                                size_t disp_pitch_bytes, int rows, int cols, float baseline, float focal,
                                                void *cuda_stream);
DCMT_API int dcmt_get_initial_disparity_mat_f32_host(const float *depth, size_t depth_pitch_bytes, float *disp,
                                                     size_t disp_pitch_bytes, int rows, int cols, float baseline,
                                                     float focal);
DCMT_API int dcmt_retrieve_optimized_depth_mat_f32(const float *disp, size_t disp_pitch_bytes, float *depth,
                                                   size_t depth_pitch_bytes, int rows, int cols, float baseline,
                                                   float focal, float depth_clip, void *cuda_stream);
DCMT_API int dcmt_retrieve_optimized_depth_mat_f32_host(const float *disp, size_t disp_pitch_bytes, float *depth,
                                                        size_t depth_pitch_bytes, int rows, int cols, float baseline,
                                                        float focal, float depth_clip);

/* (8f #3) evaluation reductions: replace evaluate_performance (src/DC_lidar_only/main.cpp:16-34, mode
 * DCMT_EVAL_GT_VALID: pixels with gt > tolerance, result mean_err = sum(gt - r) / count, which that program calls
 * "mse"), evaluate_performance (src/DC_lidar_camera/main_lc.cpp:85-116) and evaluate_performances
 * (src/DC_stereo_lidar/main_sl.cpp:1031-1061) (mode DCMT_EVAL_BOTH_VALID: pixels with gt > tolerance and
 * r > tolerance; rmse = sqrt(sum d^2 / count), mae = sum |d| / count).  `tolerance` is the reference's `int tolerance`
 * converted to float: 0 for main.cpp (`= 0`) and main_lc.cpp (`= 0.1` truncates), 2 for main_sl.cpp.  One result per
 * frame.  Sums are accumulated in double in a fixed order (deterministic; the reference accumulates in float32 in
 * raster order, so its own figures differ from the exact sums in the 4th-5th digit).  An empty mask gives NaN like
 * the reference's 0 / 0. */
enum { DCMT_EVAL_GT_VALID = 0, DCMT_EVAL_BOTH_VALID = 1 };
typedef struct dcmt_eval_result {
    double count, sum_err, sum_abs, sum_sq;
    float mean_err, mae, rmse;
    int32_t pad;
} dcmt_eval_result;
DCMT_API int dcmt_evaluate_f32(const float *gt, const float *dense, int rows, int cols, size_t pitch_bytes,
                               size_t frame_stride_bytes, int n_frames, float tolerance, int mode,
                               dcmt_eval_result *results /* device, n_frames */, void *cuda_stream);
DCMT_API int dcmt_evaluate_f32_host(const float *gt, const float *dense, int rows, int cols, size_t pitch_bytes,
                                    size_t frame_stride_bytes, int n_frames, float tolerance, int mode,
                                    dcmt_eval_result *results /* host, n_frames */);
/* (8f #3, KITTI on-disk format) the same reductions on KITTI ground truth as read: the uint16 payload of the depth PNG
 * (cv::imread(..., IMREAD_ANYDEPTH); uint16 = metres * 256, 0 = no measurement) -- it replaces the GT's
 * convertTo(CV_32F, 1.0 / 256.0) of main.cpp:82 and main_lc.cpp:159-224 in front of evaluate_performance, and serves
 * evaluate_performances (main_sl.cpp:1031-1061) as well.  dcmt_evaluate_u16 scores a float32 result;
 * dcmt_evaluate_u16_u16 scores a KITTI uint16 result as well (the output of the *_u16_u16 completion calls, what a caller
 * stores as a PNG).  A uint16 value u is decoded to (float)u * (1.0f / 256.0f), which is exact; the mask test, the
 * float32 subtraction and the double accumulation are those of dcmt_evaluate_f32.  GT and result have their own pitches
 * and frame strides in bytes (0 = dense); a pitch or stride that is not a multiple of the element size or too small is
 * DCMT_E_BADARG.  Results are byte-identical to dcmt_evaluate_f32 on the decoded planes (u / 256) whenever those planes
 * have the same pitch, frame stride and base alignment counted in elements (the 4-pixel vector loads are taken under
 * the same condition).  HBM traffic is 6 (u16 GT, float32 result) or 4 (both uint16) bytes per pixel instead of 8, and
 * the *_host variants stage 2 + 4 or 2 + 2 bytes per pixel. */
DCMT_API int dcmt_evaluate_u16(const uint16_t *gt_u16, const float *dense, int rows, int cols, size_t gt_pitch_bytes,
                               size_t gt_frame_stride_bytes, size_t dense_pitch_bytes, size_t dense_frame_stride_bytes,
                               int n_frames, float tolerance, int mode, dcmt_eval_result *results /* device, n_frames */,
                               void *cuda_stream);
DCMT_API int dcmt_evaluate_u16_host(const uint16_t *gt_u16, const float *dense, int rows, int cols, size_t gt_pitch_bytes,
                                    size_t gt_frame_stride_bytes, size_t dense_pitch_bytes, size_t dense_frame_stride_bytes,
                                    int n_frames, float tolerance, int mode, dcmt_eval_result *results /* host, n_frames */);
DCMT_API int dcmt_evaluate_u16_u16(const uint16_t *gt_u16, const uint16_t *dense_u16, int rows, int cols, size_t gt_pitch_bytes,
                                   size_t gt_frame_stride_bytes, size_t dense_pitch_bytes, size_t dense_frame_stride_bytes,
                                   int n_frames, float tolerance, int mode, dcmt_eval_result *results /* device, n_frames */,
                                   void *cuda_stream);
DCMT_API int dcmt_evaluate_u16_u16_host(const uint16_t *gt_u16, const uint16_t *dense_u16, int rows, int cols,
                                        size_t gt_pitch_bytes, size_t gt_frame_stride_bytes, size_t dense_pitch_bytes,
                                        size_t dense_frame_stride_bytes, int n_frames, float tolerance, int mode,
                                        dcmt_eval_result *results /* host, n_frames */);

/* The figures the KITTI depth-completion benchmark publishes: MAE and RMSE in mm, iMAE and iRMSE in 1/km, over every
 * pixel with ground truth after the prediction's holes are filled by the devkit's background interpolation.  The rule
 * below restates the devkit's interpolateBackground and per-image error loop; the tests pin the library to a numpy
 * restatement of this text, not to the devkit itself.  Per frame, with g the GT and p the prediction in metres:
 *  1. A uint16 value u decodes to (float)u * (1.0f / 256.0f).  g is valid iff g > 0, p iff p > 0 (so uint16 0, float32 0,
 *     negatives and NaN are invalid).
 *  2. Background interpolation of p.  Row pass: in each row, an invalid pixel takes min(L, R) of the values of the nearest
 *     valid pixels to its left and right in that row, or the one that exists; a row with no valid pixel stays invalid.
 *     Column pass: with F / B the first / last rows holding a valid p, every pixel of a row above F takes the row-pass
 *     value of its column in row F, every pixel of a row below B that of row B.  Invalid rows strictly between F and B,
 *     and every pixel of a frame with no valid p, stay unfilled and carry the devkit's marker p = -1.
 *  3. At GT-valid pixels only: e = fabsf(g - p) (float32, then widened to double), ie = fabs(1.0 / g - 1.0 / p) in double.
 *  4. Sums in double, combined in a fixed order: n_gt (GT-valid pixels), n_pred (of those, valid in p before the
 *     interpolation), n_unfilled (left unfilled by step 2), sum_abs = sum e, sum_sq = sum e^2, sum_iabs = sum ie,
 *     sum_isq = sum ie^2.
 *  5. mae_mm = 1000 * sum_abs / n_gt, rmse_mm = 1000 * sqrt(sum_sq / n_gt), imae_per_km = 1000 * sum_iabs / n_gt,
 *     irmse_per_km = 1000 * sqrt(sum_isq / n_gt), density = n_pred / n_gt; each computed in double and rounded once to
 *     float; NaN when n_gt == 0.
 * One record per frame; the benchmark reports the mean of the per-image figures over the set, which the caller takes.
 * Type pairs, pitches and frame strides (bytes per side, 0 = dense) are those of dcmt_evaluate_u16[_u16] plus a float32
 * pair; a uint16 call gives the bytes of the float32 call on the decoded planes laid out alike in elements.  The pixels of
 * a valid prediction are visited in the order of dcmt_evaluate_*, so on a prediction with no invalid pixel n_gt, sum_abs
 * and sum_sq are byte-equal to count, sum_abs and sum_sq of dcmt_evaluate_* in mode DCMT_EVAL_GT_VALID with tolerance 0.
 * Bad arguments return DCMT_E_BADARG before any device work; n_frames == 0 is a no-op. */
typedef struct dcmt_kitti_metrics {
    double n_gt, n_pred, n_unfilled;
    double sum_abs, sum_sq, sum_iabs, sum_isq;
    float mae_mm, rmse_mm, imae_per_km, irmse_per_km, density;
    int32_t pad;
} dcmt_kitti_metrics;
DCMT_API int dcmt_evaluate_kitti_f32(const float *gt, const float *pred, int rows, int cols, size_t gt_pitch_bytes,
                                     size_t gt_frame_stride_bytes, size_t pred_pitch_bytes, size_t pred_frame_stride_bytes,
                                     int n_frames, dcmt_kitti_metrics *results /* device, n_frames */, void *cuda_stream);
DCMT_API int dcmt_evaluate_kitti_f32_host(const float *gt, const float *pred, int rows, int cols, size_t gt_pitch_bytes,
                                          size_t gt_frame_stride_bytes, size_t pred_pitch_bytes, size_t pred_frame_stride_bytes,
                                          int n_frames, dcmt_kitti_metrics *results /* host, n_frames */);
DCMT_API int dcmt_evaluate_kitti_u16(const uint16_t *gt_u16, const float *pred, int rows, int cols, size_t gt_pitch_bytes,
                                     size_t gt_frame_stride_bytes, size_t pred_pitch_bytes, size_t pred_frame_stride_bytes,
                                     int n_frames, dcmt_kitti_metrics *results /* device, n_frames */, void *cuda_stream);
DCMT_API int dcmt_evaluate_kitti_u16_host(const uint16_t *gt_u16, const float *pred, int rows, int cols, size_t gt_pitch_bytes,
                                          size_t gt_frame_stride_bytes, size_t pred_pitch_bytes, size_t pred_frame_stride_bytes,
                                          int n_frames, dcmt_kitti_metrics *results /* host, n_frames */);
DCMT_API int dcmt_evaluate_kitti_u16_u16(const uint16_t *gt_u16, const uint16_t *pred_u16, int rows, int cols,
                                         size_t gt_pitch_bytes, size_t gt_frame_stride_bytes, size_t pred_pitch_bytes,
                                         size_t pred_frame_stride_bytes, int n_frames,
                                         dcmt_kitti_metrics *results /* device, n_frames */, void *cuda_stream);
DCMT_API int dcmt_evaluate_kitti_u16_u16_host(const uint16_t *gt_u16, const uint16_t *pred_u16, int rows, int cols,
                                              size_t gt_pitch_bytes, size_t gt_frame_stride_bytes, size_t pred_pitch_bytes,
                                              size_t pred_frame_stride_bytes, int n_frames,
                                              dcmt_kitti_metrics *results /* host, n_frames */);

/* (8f #2) LiDAR projection + normalisation: replaces the loops of src/DC_stereo_lidar/main_sl.cpp:478-523 (withSuperPixels;
 * the same code in vedi_pc :340-385): Velodyne points (n_points x 4 float32: x, y, z, intensity -- the .bin payload)
 * -> T (4x4, velodyne to camera; rows 0..2 used) -> keep z > 0 -> P (3x4) -> perspective division -> bounds test ->
 * (int) truncation -> depth scatter where the LAST point in file order wins -> cv::normalize(NORM_MINMAX, norm_a,
 * norm_b) (the reference uses 0, 80).  T and P are HOST pointers, row-major (Eigen's default storage is column-major:
 * pass the transpose or use the C++ shim).  `projected` receives the sparse depth image (main_sl.cpp's
 * projected_depths, 0 = empty), `normalized` the normalised one (the input of interpolate_with_superpixels); either may
 * be NULL.  `n_projected` (int32, optional) counts the points that landed in the image (:508).  Float arithmetic
 * follows the source order without FMA contraction; the result is deterministic. */
DCMT_API int dcmt_lidar_project_f32(const float *points, int n_points, const float *T_host, const float *P_host, int rows,
                                    int cols, float *projected_or_null, float *normalized_or_null, float norm_a,
                                    float norm_b, int32_t *n_projected_or_null, void *cuda_stream);
/* the same for a batch of clouds in four launches (one cloud alone is launch bound): cloud c holds n_points_dev[c] points
 * (DEVICE array of n_clouds int32; NULL: max_points each) at points + c * cloud_stride_points * 4 floats; max_points bounds
 * every count.  Outputs are n_clouds planes (n_projected: n_clouds int32); one T and P for the whole batch. */
DCMT_API int dcmt_lidar_project_batch_f32(const float *points, const int32_t *n_points_dev_or_null, int max_points,
                                          size_t cloud_stride_points, int n_clouds, const float *T_host, const float *P_host,
                                          int rows, int cols, float *projected_or_null, float *normalized_or_null, float norm_a,
                                          float norm_b, int32_t *n_projected_or_null, void *cuda_stream);
DCMT_API int dcmt_lidar_project_f32_host(const float *points, int n_points, const float *T_host, const float *P_host,
                                         int rows, int cols, float *projected_or_null, float *normalized_or_null,
                                         float norm_a, float norm_b, int32_t *n_projected_or_null);

/* (8f #1) SLIC superpixels: replaces Slic::generate_superpixels(cv::Mat& lab_image, int step, int nc)
 * (src/DC_lidar_camera/slic.cpp:101-182, with init_data :19-59, find_local_minimum :72-99, compute_dist :61-69), the
 * producer of the label map of interpolate_with_superpixels.  `lab` is the CV_8UC3 image after
 * cv::cvtColor(COLOR_BGR2Lab) (main_lc.cpp:184, rows x cols x 3 bytes, continuous); `step` the already truncated int
 * (the reference passes a double into an int parameter, main_lc.cpp:197-201), `nc` the colour weight, `iterations` the
 * reference's NR_ITERATIONS = 10 (slic.h:20).  `labels` receives Slic::clusters as row-major int32 [row][col] (the
 * layout dcmt_interpolate_with_superpixels_f32 takes; -1 = never assigned), `centers_or_null` the final
 * Slic::centers (n_centers x 5 doubles: L, a, b, x, y; NaN for an empty cluster like the reference's 0 / 0).
 * dcmt_slic_center_count gives slic.centers.size() for a shape.  Labels are bit-identical to a scalar build of the
 * reference (same double arithmetic, ties to the lowest centre index, stale labels kept).  Needs step >= 4 (below
 * that the reference itself reads outside the image in find_local_minimum).  `n_frames` images (contiguous, each
 * rows x cols x 3) are segmented side by side: labels n_frames x rows x cols, centers n_frames x n_centers x 5. */
DCMT_API int dcmt_slic_center_count(int rows, int cols, int step);
DCMT_API int dcmt_slic_u8c3(const uint8_t *lab, int rows, int cols, int n_frames, int step, int nc, int iterations,
                            int32_t *labels, double *centers_or_null, void *cuda_stream);
DCMT_API int dcmt_slic_u8c3_host(const uint8_t *lab, int rows, int cols, int n_frames, int step, int nc, int iterations,
                                 int32_t *labels, double *centers_or_null);
/* the pair cv::cvtColor(img, lab, COLOR_BGR2Lab) + slic.generate_superpixels(lab, step, nc) in one call, from the
 * CV_8UC3 BGR image as read (main_lc.cpp:182-201; main_sl.cpp:438-450 with 100 superpixels and nc = 40): the Lab
 * frames are made by dcmt_bgr2lab_u8 inside the workspace of (device, stream) and segmented as by dcmt_slic_u8c3, so
 * labels and centres equal dcmt_slic_u8c3 on OpenCV's Lab.  Arguments as for dcmt_slic_u8c3 with `bgr` (contiguous,
 * n_frames x rows x cols x 3) in place of `lab`; a host caller moves 3 bytes per pixel in and the labels out. */
DCMT_API int dcmt_slic_bgr_u8c3(const uint8_t *bgr, int rows, int cols, int n_frames, int step, int nc, int iterations,
                                int32_t *labels, double *centers_or_null, void *cuda_stream);
DCMT_API int dcmt_slic_bgr_u8c3_host(const uint8_t *bgr, int rows, int cols, int n_frames, int step, int nc, int iterations,
                                     int32_t *labels, double *centers_or_null);

/* debugging aid: runs the generic pipeline on ONE frame and snapshots intermediate images
 * (device memory, n_stages * rows * cols floats, stage order of oracle/dcmt_oracle.c; stages the
 * kernels never materialise are left untouched).  `stage_mask_out` (host) gets a bit per stage written. */
DCMT_API int dcmt_img_completion_stages_f32(const float *sparse, float *dense, int rows, int cols, int blur_type,
                                            float *stages, int n_stages, uint32_t *stage_mask_out,
                                            void *cuda_stream);

/* debugging aid: runs the fused strict-q8 kernels on one chunk of frames (device pointers, contiguous) and records
 * 16 clock64() stamps per CTA at the phase boundaries of k_q8_front / k_q8_tail (device arrays of
 * tiles_per_frame * n_frames * 16 int64 each; use ceil(rows/32)*ceil(cols/32) tiles as an upper bound). */
DCMT_API int dcmt_debug_q8_phase_cycles(const float *sparse, float *dense, int rows, int cols, int n_frames,
                                        long long *front_stamps, long long *tail_stamps, int *tiles_per_frame,
                                        void *cuda_stream);

#ifdef __cplusplus
}
#endif
#endif /* DCMT_H_ */
