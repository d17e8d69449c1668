// common.cuh -- shared definitions for the dcmt CUDA kernels (sm_100a).
#pragma once
#include <cfloat>
#include <cstddef>
#include <cstdint>
#ifdef DCMT_EMU
// CPU emulation of the CUDA execution model, tests only (tests/emu/cuda_emu.h); never defined for libdcmt.so
#include "cuda_emu.h"
#include <cstring>
#else
#include <cuda.h>  // CUtensorMap and its enums only; the encoder is fetched with cudaGetDriverEntryPoint (no -lcuda)
#include <cuda_runtime.h>
#define DCMT_DYN_SMEM(type, name)                                         \
    extern __shared__ __align__(128) unsigned char dcmt_dyn_smem_raw[];   \
    type* name = reinterpret_cast<type*>(dcmt_dyn_smem_raw)
namespace dcmt { void note_launch(); }  // launch counter behind dcmt_launch_count() (api.cu)
#define DCMT_LAUNCH(kernel, grid, block, smem, stream, ...) \
    (dcmt::note_launch(), kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__))
#endif

namespace dcmt {

// ---- TMA (cp.async.bulk.tensor) tile load of a uint16 or float32 plane: one thread issues one 3-D box copy (columns,
// rows, frame) global -> shared; elements of the box outside the tensor are ZERO-filled by the hardware, the copy signals
// an mbarrier with its byte count.  A map cannot be encoded (an error is returned) unless the base, the row pitch and
// the frame stride are multiples of 16 bytes.  The emulator build replaces the map by a plain description, refuses
// the same layouts and copies in place.
#ifdef DCMT_EMU
struct TensorMap3D {
    const void* base;
    int elem;           // bytes per element
    int dim[3];         // elements: columns, rows, frames
    size_t stride[2];   // bytes between rows, between frames
    int box[2];         // columns, rows of the box (one frame)
};
inline cudaError_t tma_encode_3d(TensorMap3D* m, const void* base, int elem, int cols, int rows, int frames, size_t row_bytes,
                                 size_t frame_bytes, int box_cols, int box_rows) {
    if (box_cols > 256 || box_rows > 256 || (row_bytes & 15) || (frame_bytes & 15) || (reinterpret_cast<uintptr_t>(base) & 15))
        return cudaErrorInvalidValue;
    *m = TensorMap3D{base, elem, {cols, rows, frames}, {row_bytes, frame_bytes}, {box_cols, box_rows}};
    return cudaSuccess;
}
inline cudaError_t tma_encode_u16_3d(TensorMap3D* m, const uint16_t* base, int cols, int rows, int frames, size_t row_bytes,
                                     size_t frame_bytes, int box_cols, int box_rows) {
    return tma_encode_3d(m, base, 2, cols, rows, frames, row_bytes, frame_bytes, box_cols, box_rows);
}
inline cudaError_t tma_encode_f32_3d(TensorMap3D* m, const float* base, int cols, int rows, int frames, size_t row_bytes,
                                     size_t frame_bytes, int box_cols, int box_rows) {
    return tma_encode_3d(m, base, 4, cols, rows, frames, row_bytes, frame_bytes, box_cols, box_rows);
}
inline void tma_bar_init(uint64_t*) {}
inline void tma_load_3d(void* smem_dst, const TensorMap3D* m, int c0, int c1, int c2, uint64_t*, uint32_t) {
    char* d = static_cast<char*>(smem_dst);
    for (int r = 0; r < m->box[1]; ++r)
        for (int c = 0; c < m->box[0]; ++c) {
            const int x = c0 + c, y = c1 + r;
            const bool in = x >= 0 && x < m->dim[0] && y >= 0 && y < m->dim[1] && c2 >= 0 && c2 < m->dim[2];
            char* o = d + ((size_t)r * m->box[0] + c) * m->elem;
            if (in) std::memcpy(o, static_cast<const char*>(m->base) + (size_t)c2 * m->stride[1] + (size_t)y * m->stride[0] + (size_t)x * m->elem, m->elem);
            else std::memset(o, 0, m->elem);
        }
}
inline void tma_bar_wait(uint64_t*, uint32_t) {}
#else
typedef CUtensorMap TensorMap3D;
cudaError_t tma_encode_u16_3d(TensorMap3D* m, const uint16_t* base, int cols, int rows, int frames, size_t row_bytes,
                              size_t frame_bytes, int box_cols, int box_rows);  // fused_q8.cu
cudaError_t tma_encode_f32_3d(TensorMap3D* m, const float* base, int cols, int rows, int frames, size_t row_bytes,
                              size_t frame_bytes, int box_cols, int box_rows);  // fused_q8.cu
__device__ __forceinline__ void tma_bar_init(uint64_t* bar) {  // one thread; follow with __syncthreads()
    const unsigned b = (unsigned)__cvta_generic_to_shared(bar);
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(b) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const TensorMap3D* m, int c0, int c1, int c2, uint64_t* bar, uint32_t bytes) {
    const unsigned b = (unsigned)__cvta_generic_to_shared(bar), d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(b), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(d),
                 "l"(reinterpret_cast<uint64_t>(m)), "r"(b), "r"(c0), "r"(c1), "r"(c2)
                 : "memory");
}
__device__ __forceinline__ void tma_bar_wait(uint64_t* bar, uint32_t parity) {
    const unsigned b = (unsigned)__cvta_generic_to_shared(bar);
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "DCMT_TMA_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DCMT_TMA_DONE;\n"
        "bra DCMT_TMA_WAIT;\n"
        "DCMT_TMA_DONE:\n"
        "}" ::"r"(b),
        "r"(parity)
        : "memory");
}
#endif

// x / n for x * n < 2^32 with magic = floor(2^32 / n) + 1 (computed on the host): one IMAD.HI instead of a division
__device__ __forceinline__ int fast_div(int x, uint32_t magic) { return (int)__umulhi((uint32_t)x, magic); }

// img_completion.cpp:59,96,113,140,154,184,194 compare float against the double literal 0.1:
//   (double)d > 0.1  <=>  d >= 0.1f      (valid pixel)
//   (double)d < 0.1  <=>  d <  0.1f      (hole)
// 0.1f is the float immediately above the real number 0.1, so the two predicates are exact complements.
__device__ __forceinline__ bool is_valid(float d) { return d >= 0.1f; }
__device__ __forceinline__ bool is_hole(float d) { return d < 0.1f; }

constexpr float kMaxDepth = 100.0f;  // img_completion.cpp:23
constexpr float kAbsentMax = -FLT_MAX;  // OpenCV morphologyDefaultBorderValue for dilate
constexpr float kAbsentMin = FLT_MAX;   // ... and for erode

// img_completion.cpp:55-67 / :191-202
__device__ __forceinline__ float invert_valid(float d) { return is_valid(d) ? kMaxDepth - d : d; }

// cv::borderInterpolate(p, len, BORDER_REFLECT_101)
__device__ __forceinline__ int reflect101(int p, int len) {
    if (len == 1) return 0;
    while (p < 0 || p >= len) p = p < 0 ? -p : 2 * len - 2 - p;
    return p;
}

__device__ __forceinline__ int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

// per-frame counters kept in the workspace (int32 each)
struct FrameCounters {
    int holes_after_extrapolation;  // counted by the first 31x31 fill before filling (stats[2])
    int holes_after_first_fill;     // left after the first 31x31 fill (stats[1])
    int holes_remaining;            // != 0 only if the fill loop hit its pass bound
    int extra_passes;               // effective passes after the first fill
    int path;                       // 0 generic, 1 fused q8
    int needs_generic;              // fused kernel could not finish this frame
    int pad[2];
};

// plain description of a batch of row-major float frames
struct Batch {
    int rows, cols, n_frames;
    size_t pitch;         // elements between rows
    size_t frame_stride;  // elements between frames
};

}  // namespace dcmt
