// color.cu -- cv::cvtColor(COLOR_BGR2Lab) on 8-bit images, the conversion in front of Slic::generate_superpixels
// (main_lc.cpp:182-184, main_sl.cpp:438).
//
//   k_bgr2lab   OpenCV's 8-bit path (RGB2Lab_b): sRGB gamma by table, fixed-point XYZ with 12-bit coefficients, the Lab
//               cube root by table, fixed-point L, a, b with 15-bit scaling.  Bit-equal to cv2 4.13 on all 2^24 colours.
//
// The tables (lab_tables.cuh) are generated and checked against cv2 by oracle/make_lab_tables.py.  Each block copies them
// to shared memory (4.6 KB): lanes index them with data-dependent, divergent indices, which constant memory would
// serialise.
#include "color.cuh"
#include "lab_tables.cuh"

namespace dcmt {
namespace {

constexpr int kThreads = 256;
constexpr int kPx = 16;  // pixels per thread: 48 bytes, three 16-byte loads and three 16-byte stores

// one pixel: (B, G, R) bytes -> L | a << 8 | b << 16
__device__ __forceinline__ unsigned lab_pixel(const uint16_t* G, const uint16_t* C, unsigned b, unsigned g, unsigned r) {
    const int gb = G[b], gg = G[g], gr = G[r];
    // rows X, Y, Z of sRGB -> XYZ / white point * 4096, applied to (R, G, B); every index is at most 2040
    const int fX = C[(1777 * gr + 1541 * gg + 778 * gb + 2048) >> 12];
    const int fY = C[(871 * gr + 2929 * gg + 296 * gb + 2048) >> 12];
    const int fZ = C[(73 * gr + 448 * gg + 3575 * gb + 2048) >> 12];
    const int L = (296 * fY - 1336934 + 16384) >> 15;  // arithmetic shifts, as OpenCV's CV_DESCALE on int
    const int A = (500 * (fX - fY) + 128 * 32768 + 16384) >> 15;
    const int B = (200 * (fY - fZ) + 128 * 32768 + 16384) >> 15;
    return (unsigned)clampi(L, 0, 255) | (unsigned)clampi(A, 0, 255) << 8 | (unsigned)clampi(B, 0, 255) << 16;
}

// One thread converts kPx consecutive pixels of a row; blockIdx.z = frame, the (row, pixel group) pairs of the frame
// are strided over the blocks of x.  Groups that end inside the row and are 16-byte aligned at both ends take the vector
// path; ragged row ends and unaligned rows go pixel by pixel.
__global__ void __launch_bounds__(kThreads) k_bgr2lab(const uint8_t* __restrict__ bgr, size_t bgr_pitch, size_t bgr_fstride,
                                                      uint8_t* __restrict__ lab, size_t lab_pitch, size_t lab_fstride, int rows,
                                                      int cols) {
    __shared__ uint16_t sG[kLabGammaSize];
    __shared__ uint16_t sC[kLabCbrtSize];
    for (int i = threadIdx.x; i < kLabGammaSize; i += kThreads) sG[i] = kLabGamma[i];
    for (int i = threadIdx.x; i < kLabCbrtSize; i += kThreads) sC[i] = kLabCbrt[i];
    __syncthreads();
    const unsigned groups = (unsigned)(cols + kPx - 1) / kPx, total = (unsigned)rows * groups;  // < 2^31 (api.cu)
    const uint8_t* fsrc = bgr + (size_t)blockIdx.z * bgr_fstride;
    uint8_t* fdst = lab + (size_t)blockIdx.z * lab_fstride;
    for (unsigned i = blockIdx.x * kThreads + threadIdx.x; i < total; i += gridDim.x * kThreads) {
        const unsigned r = i / groups, c0 = (i - r * groups) * kPx;
        const uint8_t* src = fsrc + (size_t)r * bgr_pitch + (size_t)c0 * 3;
        uint8_t* dst = fdst + (size_t)r * lab_pitch + (size_t)c0 * 3;
        if (c0 + kPx <= (unsigned)cols && ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15) == 0) {
            const uint4 v0 = __ldg(reinterpret_cast<const uint4*>(src)), v1 = __ldg(reinterpret_cast<const uint4*>(src) + 1),
                        v2 = __ldg(reinterpret_cast<const uint4*>(src) + 2);
            const unsigned w[12] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w, v2.x, v2.y, v2.z, v2.w};
            unsigned o[12] = {};
#pragma unroll
            for (int j = 0; j < kPx; ++j) {
                unsigned px[3];
#pragma unroll
                for (int c = 0; c < 3; ++c) px[c] = (w[(3 * j + c) >> 2] >> (8 * ((3 * j + c) & 3))) & 255u;
                const unsigned v = lab_pixel(sG, sC, px[0], px[1], px[2]);
#pragma unroll
                for (int c = 0; c < 3; ++c) o[(3 * j + c) >> 2] |= ((v >> (8 * c)) & 255u) << (8 * ((3 * j + c) & 3));
            }
            uint4* d4 = reinterpret_cast<uint4*>(dst);
            d4[0] = make_uint4(o[0], o[1], o[2], o[3]);
            d4[1] = make_uint4(o[4], o[5], o[6], o[7]);
            d4[2] = make_uint4(o[8], o[9], o[10], o[11]);
        } else {
            const int n = cols - (int)c0 < kPx ? cols - (int)c0 : kPx;
            for (int j = 0; j < n; ++j) {
                const unsigned v = lab_pixel(sG, sC, src[3 * j], src[3 * j + 1], src[3 * j + 2]);
                dst[3 * j] = (uint8_t)v;
                dst[3 * j + 1] = (uint8_t)(v >> 8);
                dst[3 * j + 2] = (uint8_t)(v >> 16);
            }
        }
    }
}

}  // namespace

cudaError_t color_bgr2lab(const uint8_t* bgr, size_t bgr_pitch, size_t bgr_fstride, uint8_t* lab, size_t lab_pitch, size_t lab_fstride,
                          int rows, int cols, int n_frames, cudaStream_t st) {
    if (n_frames == 0) return cudaSuccess;
    const unsigned long long total = (unsigned long long)rows * ((cols + kPx - 1) / kPx);
    const unsigned one_each = (unsigned)((total + kThreads - 1) / kThreads);  // blocks for one pixel group per thread
    // eight groups per thread amortise the table copy over 128 pixels; a small batch spreads over the SMs instead
    unsigned bx = (one_each + 7) / 8;
    if ((unsigned long long)bx * n_frames < 1024) bx = one_each;
    DCMT_LAUNCH(k_bgr2lab, dim3(bx, 1, n_frames), dim3(kThreads), 0, st, bgr, bgr_pitch, bgr_fstride, lab, lab_pitch, lab_fstride, rows,
                cols);
    return cudaGetLastError();
}

}  // namespace dcmt
