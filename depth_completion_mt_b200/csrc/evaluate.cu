// evaluate.cu -- the reference's evaluation loops as device reductions (SURVEY.md 8f #3):
//   evaluate_performance   DC_lidar_only/main.cpp:16-34       mask gt > 0          mse = sum(gt - r) / count  (a signed mean)
//   evaluate_performance   DC_lidar_camera/main_lc.cpp:85-116 mask gt > 0 && r > 0 mse = sqrt(sum d^2 / count), mae = sum |d| / count
//                          (`int tolerance = 0.1` truncates to 0, :88)
//   evaluate_performances  DC_stereo_lidar/main_sl.cpp:1031-1061  the same with tolerance 2
// The reference accumulates in float32 in raster order; here every thread accumulates in double and the partial sums
// are combined in a fixed order (lanes, warps, blocks), so results are deterministic and closer to the exact sums than
// the reference's own (tests state the tolerance against the literal float32 loop).  HBM-bound: 8 bytes per pixel for
// float32 planes, 6 with a KITTI uint16 GT plane and 4 with both planes uint16 (main.cpp:82's convertTo(CV_32F, 1/256)
// happens in the load; the decoded value is exact, so the results are those of the float32 planes u / 256).
// The KITTI depth-completion benchmark's figures (MAE / RMSE in mm, iMAE / iRMSE in 1/km after the devkit's background
// interpolation of the prediction) come from the same traversal: k_kitti_first_last, k_kitti_partial, k_kitti_finish.
#include "evaluate.cuh"

namespace dcmt {
namespace {

constexpr int ET = 256;

__device__ __forceinline__ double shfl_down_double(double v, int d) {
    int lo = __shfl_down_sync(0xffffffffu, (int)(__double_as_longlong(v) & 0xffffffffll), d);
    int hi = __shfl_down_sync(0xffffffffu, (int)(__double_as_longlong(v) >> 32), d);
    return __longlong_as_double(((long long)hi << 32) | (unsigned)lo);
}

struct Acc {
    double n, e, a, s;
    __device__ __forceinline__ void add(float g, float r, float tol, int mode) {
        // `gt > tolerance` compares a float with an int in the reference: the int converts to float
        if (g > tol && (mode == 0 || r > tol)) {
            const float d = g - r;  // float subtraction as in the reference; fabs / squaring below are exact in double
            n += 1.0;
            e += (double)d;
            a += fabs((double)d);
            s += (double)d * (double)d;
        }
    }
};

// Element types of a plane: float32 metres, or KITTI uint16 = metres * 256 decoded exactly to u * 2^-8.  Vec4 is the
// vector load of the 4-pixel items: 16 bytes of float32, 8 of uint16.
template <class T>
struct Elem;
template <>
struct Elem<float> {
    using Vec4 = float4;
    static __device__ __forceinline__ float dec(float v) { return v; }
};
template <>
struct Elem<uint16_t> {
    using Vec4 = ushort4;
    static __device__ __forceinline__ float dec(uint16_t v) { return (float)v * (1.0f / 256.0f); }
};

template <class G, class R>
__global__ void __launch_bounds__(ET) k_eval_partial(const G* __restrict__ gt, const R* __restrict__ rr, int rows, int cols, size_t gpitch,
                                                     size_t gfstride, size_t rpitch, size_t rfstride, float tol, int mode, int vec_ok,
                                                     double* __restrict__ partials) {
    using EG = Elem<G>;
    using ER = Elem<R>;
    const int frame = blockIdx.y;
    const G* g0 = gt + (size_t)frame * gfstride;
    const R* r0 = rr + (size_t)frame * rfstride;
    Acc acc{0.0, 0.0, 0.0, 0.0};
    const int c4 = vec_ok ? cols / 4 : 0;
    for (int y = blockIdx.x; y < rows; y += gridDim.x) {
        const G* g = g0 + (size_t)y * gpitch;
        const R* r = r0 + (size_t)y * rpitch;
        for (int i = threadIdx.x; i < c4; i += ET) {
            const typename EG::Vec4 a = __ldg(reinterpret_cast<const typename EG::Vec4*>(g) + i);
            const typename ER::Vec4 b = __ldg(reinterpret_cast<const typename ER::Vec4*>(r) + i);
            acc.add(EG::dec(a.x), ER::dec(b.x), tol, mode);
            acc.add(EG::dec(a.y), ER::dec(b.y), tol, mode);
            acc.add(EG::dec(a.z), ER::dec(b.z), tol, mode);
            acc.add(EG::dec(a.w), ER::dec(b.w), tol, mode);
        }
        for (int x = c4 * 4 + threadIdx.x; x < cols; x += ET) acc.add(EG::dec(__ldg(g + x)), ER::dec(__ldg(r + x)), tol, mode);
    }
    // lanes -> warps -> block, always in the same order
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) {
        acc.n += shfl_down_double(acc.n, d);
        acc.e += shfl_down_double(acc.e, d);
        acc.a += shfl_down_double(acc.a, d);
        acc.s += shfl_down_double(acc.s, d);
    }
    __shared__ double sm[ET / 32][4];
    const int warp = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) {
        sm[warp][0] = acc.n;
        sm[warp][1] = acc.e;
        sm[warp][2] = acc.a;
        sm[warp][3] = acc.s;
    }
    __syncthreads();
    if (threadIdx.x < 4) {
        double t = 0.0;
        for (int w = 0; w < ET / 32; ++w) t += sm[w][threadIdx.x];
        partials[((size_t)frame * gridDim.x + blockIdx.x) * 4 + threadIdx.x] = t;
    }
}

__global__ void k_eval_finish(const double* __restrict__ partials, int nblocks, int n_frames, EvalResult* __restrict__ out) {
    const int frame = blockIdx.x * blockDim.x + threadIdx.x;
    if (frame >= n_frames) return;
    double t[4] = {0.0, 0.0, 0.0, 0.0};
    for (int b = 0; b < nblocks; ++b)
        for (int k = 0; k < 4; ++k) t[k] += partials[((size_t)frame * nblocks + b) * 4 + k];
    EvalResult r;
    r.count = t[0];
    r.sum_err = t[1];
    r.sum_abs = t[2];
    r.sum_sq = t[3];
    // 0 / 0 = NaN for an empty mask, like the reference's float division
    r.mean_err = (float)(t[1] / t[0]);
    r.mae = (float)(t[2] / t[0]);
    r.rmse = (float)sqrt(t[3] / t[0]);
    r.pad = 0;
    out[frame] = r;
}

// 4-pixel items need every row and frame of both planes to start on a 4-element boundary
template <class T>
bool vec4_ok(const T* p, size_t pitch, size_t fstride) {
    return pitch % 4 == 0 && fstride % 4 == 0 && reinterpret_cast<uintptr_t>(p) % (4 * sizeof(T)) == 0;
}

// ---- the KITTI depth-completion benchmark's figures (dcmt_kitti_metrics in include/dcmt.h).  The prediction's holes are
// filled as the devkit's background interpolation does: within a row, min of the nearest valid values to the left and
// right (or the one that exists); rows above the first / below the last row holding a valid value take that row's
// filled values; everything else stays unfilled at -1.  Only GT-valid pixels the prediction missed look at their
// neighbours, so a dense prediction is read once, in the pixel order of k_eval_partial.
constexpr int kKittiSmemWords = 8192;  // validity bits of rows up to 262 144 columns fit in 32 KB of shared memory
constexpr int kKittiSums = 7;

// the first and the last row of each frame holding a valid prediction (-1, -1 for none), reading rows from each end
// only until one holds a valid pixel
template <class R>
__global__ void __launch_bounds__(ET) k_kitti_first_last(const R* __restrict__ rr, int rows, int cols, size_t rpitch, size_t rfstride,
                                                         int32_t* __restrict__ first_last) {
    const R* r0 = rr + (size_t)blockIdx.x * rfstride;
    int first = -1, last = -1;
    for (int y = 0; y < rows && first < 0; ++y) {
        int any = 0;
        for (int x = threadIdx.x; x < cols && !any; x += ET) any = Elem<R>::dec(__ldg(r0 + (size_t)y * rpitch + x)) > 0.0f;
        if (__syncthreads_or(any)) first = y;
    }
    for (int y = rows - 1; first >= 0 && y >= first && last < 0; --y) {
        int any = 0;
        for (int x = threadIdx.x; x < cols && !any; x += ET) any = Elem<R>::dec(__ldg(r0 + (size_t)y * rpitch + x)) > 0.0f;
        if (__syncthreads_or(any)) last = y;
    }
    if (threadIdx.x == 0) {
        first_last[2 * blockIdx.x] = first;
        first_last[2 * blockIdx.x + 1] = last;
    }
}

struct KittiAcc {
    double n, np, nu, a, s, ia, is;
    // the error terms of a GT-valid pixel whose (filled) prediction is p; p = -1 when unfilled
    __device__ __forceinline__ void term(float g, float p) {
        const float e = fabsf(g - p);  // float subtraction as in k_eval_partial; squaring is exact in double
        a += (double)e;
        s += (double)e * (double)e;
        const double ie = fabs(1.0 / (double)g - 1.0 / (double)p);
        ia += ie;
        is += ie * ie;
    }
    // a pixel as read; returns 1 for a GT-valid pixel the prediction missed (filled in a second pass over the row)
    __device__ __forceinline__ int add(float g, float p) {
        if (!(g > 0.0f)) return 0;
        n += 1.0;
        if (!(p > 0.0f)) return 1;
        np += 1.0;
        term(g, p);
        return 0;
    }
};

// the row pass at column x of `row`, whose validity bits are `bits` (`words` words, zero past the last column): the value
// at x when valid, else min(L, R) of the nearest valid values to the left and right, else the one that exists; -1 when
// the row holds none
template <class R>
__device__ __forceinline__ float row_fill(const unsigned* bits, int words, const R* __restrict__ row, int x) {
    const int w = x >> 5, b = x & 31;
    if (bits[w] >> b & 1u) return Elem<R>::dec(__ldg(row + x));
    int l = -1, r = -1;
    unsigned m = bits[w] & ((1u << b) - 1u);
    for (int k = w;;) {
        if (m) {
            l = k * 32 + 31 - __clz((int)m);
            break;
        }
        if (--k < 0) break;
        m = bits[k];
    }
    m = bits[w] & ~((2u << b) - 1u);  // 2u << 31 == 0: no bits above column 31
    for (int k = w;;) {
        if (m) {
            r = k * 32 + __ffs((int)m) - 1;
            break;
        }
        if (++k >= words) break;
        m = bits[k];
    }
    if (l < 0 && r < 0) return -1.0f;
    if (l < 0) return Elem<R>::dec(__ldg(row + r));
    if (r < 0) return Elem<R>::dec(__ldg(row + l));
    return fminf(Elem<R>::dec(__ldg(row + l)), Elem<R>::dec(__ldg(row + r)));
}

// k_eval_partial's blocks, pixel order and reductions with the KITTI terms.  `gbits` (nullptr: shared memory) holds one
// row of validity bits per block for rows wider than kKittiSmemWords words.
template <class G, class R>
__global__ void __launch_bounds__(ET) k_kitti_partial(const G* __restrict__ gt, const R* __restrict__ rr, int rows, int cols, size_t gpitch,
                                                      size_t gfstride, size_t rpitch, size_t rfstride, int vec_ok,
                                                      const int32_t* __restrict__ first_last, unsigned* __restrict__ gbits,
                                                      double* __restrict__ partials) {
    using EG = Elem<G>;
    using ER = Elem<R>;
    const int frame = blockIdx.y;
    const G* g0 = gt + (size_t)frame * gfstride;
    const R* r0 = rr + (size_t)frame * rfstride;
    const int words = (cols + 31) >> 5;
    DCMT_DYN_SMEM(unsigned, sbits);
    unsigned* bits = gbits ? gbits + ((size_t)frame * gridDim.x + blockIdx.x) * words : sbits;
    const int first = first_last[2 * frame], last = first_last[2 * frame + 1];
    KittiAcc acc{0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    const int c4 = vec_ok ? cols / 4 : 0;
    for (int y = blockIdx.x; y < rows; y += gridDim.x) {
        const G* g = g0 + (size_t)y * gpitch;
        const R* r = r0 + (size_t)y * rpitch;
        int need = 0;
        for (int i = threadIdx.x; i < c4; i += ET) {
            const typename EG::Vec4 a = __ldg(reinterpret_cast<const typename EG::Vec4*>(g) + i);
            const typename ER::Vec4 b = __ldg(reinterpret_cast<const typename ER::Vec4*>(r) + i);
            need |= acc.add(EG::dec(a.x), ER::dec(b.x));
            need |= acc.add(EG::dec(a.y), ER::dec(b.y));
            need |= acc.add(EG::dec(a.z), ER::dec(b.z));
            need |= acc.add(EG::dec(a.w), ER::dec(b.w));
        }
        for (int x = c4 * 4 + threadIdx.x; x < cols; x += ET) need |= acc.add(EG::dec(__ldg(g + x)), ER::dec(__ldg(r + x)));
        // (also the barrier that keeps the previous row's second pass from reading bits this row rewrites)
        if (!__syncthreads_or(need)) continue;
        // the row pass runs on this row, or on the first / last valid row for the rows above / below them
        const int src = y < first ? first : y > last ? last : y;
        const R* rs = r0 + (size_t)(src < 0 ? 0 : src) * rpitch;
        if (src >= 0) {
            for (int x0 = threadIdx.x & ~31; x0 < cols; x0 += ET) {
                const int x = x0 + (threadIdx.x & 31);
                const unsigned m = __ballot_sync(0xffffffffu, x < cols && ER::dec(__ldg(rs + x)) > 0.0f);
                if ((threadIdx.x & 31) == 0) bits[x0 >> 5] = m;
            }
        }
        __syncthreads();
        for (int x = threadIdx.x; x < cols; x += ET) {
            const float gv = EG::dec(__ldg(g + x));
            if (!(gv > 0.0f) || ER::dec(__ldg(r + x)) > 0.0f) continue;
            const float p = src >= 0 ? row_fill(bits, words, rs, x) : -1.0f;
            if (p < 0.0f) acc.nu += 1.0;
            acc.term(gv, p);
        }
    }
    // lanes -> warps -> block, in the order of k_eval_partial
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) {
        acc.n += shfl_down_double(acc.n, d);
        acc.np += shfl_down_double(acc.np, d);
        acc.nu += shfl_down_double(acc.nu, d);
        acc.a += shfl_down_double(acc.a, d);
        acc.s += shfl_down_double(acc.s, d);
        acc.ia += shfl_down_double(acc.ia, d);
        acc.is += shfl_down_double(acc.is, d);
    }
    __shared__ double sm[ET / 32][kKittiSums];
    const int warp = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) {
        sm[warp][0] = acc.n;
        sm[warp][1] = acc.np;
        sm[warp][2] = acc.nu;
        sm[warp][3] = acc.a;
        sm[warp][4] = acc.s;
        sm[warp][5] = acc.ia;
        sm[warp][6] = acc.is;
    }
    __syncthreads();
    if (threadIdx.x < kKittiSums) {
        double t = 0.0;
        for (int w = 0; w < ET / 32; ++w) t += sm[w][threadIdx.x];
        partials[((size_t)frame * gridDim.x + blockIdx.x) * kKittiSums + threadIdx.x] = t;
    }
}

__global__ void k_kitti_finish(const double* __restrict__ partials, int nblocks, int n_frames, KittiMetrics* __restrict__ out) {
    const int frame = blockIdx.x * blockDim.x + threadIdx.x;
    if (frame >= n_frames) return;
    double t[kKittiSums] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    for (int b = 0; b < nblocks; ++b)
        for (int k = 0; k < kKittiSums; ++k) t[k] += partials[((size_t)frame * nblocks + b) * kKittiSums + k];
    KittiMetrics m;
    m.n_gt = t[0];
    m.n_pred = t[1];
    m.n_unfilled = t[2];
    m.sum_abs = t[3];
    m.sum_sq = t[4];
    m.sum_iabs = t[5];
    m.sum_isq = t[6];
    // each figure in double, rounded once; 0 / 0 = NaN when the frame has no GT
    m.mae_mm = (float)(1000.0 * (t[3] / t[0]));
    m.rmse_mm = (float)(1000.0 * sqrt(t[4] / t[0]));
    m.imae_per_km = (float)(1000.0 * (t[5] / t[0]));
    m.irmse_per_km = (float)(1000.0 * sqrt(t[6] / t[0]));
    m.density = (float)(t[1] / t[0]);
    m.pad = 0;
    out[frame] = m;
}

}  // namespace

size_t eval_partial_doubles(int n_frames) { return (size_t)n_frames * kEvalMaxBlocks * 4; }

size_t kitti_partial_doubles(int n_frames) { return (size_t)n_frames * kEvalMaxBlocks * kKittiSums; }

size_t kitti_bits_words(int rows, int cols, int n_frames) {
    const size_t words = ((size_t)cols + 31) / 32;
    if (words <= (size_t)kKittiSmemWords) return 0;
    const size_t nb = rows < kEvalMaxBlocks ? rows : kEvalMaxBlocks;
    return words * nb * (size_t)(n_frames < 65535 ? n_frames : 65535);  // reused by every launch of 65535 frames
}

template <class G, class R>
cudaError_t kitti_run(const G* gt, size_t gpitch, size_t gfstride, const R* r, size_t rpitch, size_t rfstride, int rows, int cols,
                      int n_frames, double* partials, int32_t* first_last, unsigned* bits, KittiMetrics* out, cudaStream_t st) {
    const int nb = rows < kEvalMaxBlocks ? rows : kEvalMaxBlocks;
    const int vec_ok = vec4_ok(gt, gpitch, gfstride) && vec4_ok(r, rpitch, rfstride);
    const int words = (cols + 31) / 32;
    unsigned* gbits = words > kKittiSmemWords ? bits : nullptr;
    const size_t smem = gbits ? 0 : (size_t)words * sizeof(unsigned);
    for (int f0 = 0; f0 < n_frames; f0 += 65535) {  // gridDim.y limit
        const int nf = n_frames - f0 < 65535 ? n_frames - f0 : 65535;
        DCMT_LAUNCH((k_kitti_first_last<R>), dim3(nf), dim3(ET), 0, st, r + (size_t)f0 * rfstride, rows, cols, rpitch, rfstride,
                    first_last + (size_t)f0 * 2);
        DCMT_LAUNCH((k_kitti_partial<G, R>), dim3(nb, nf), dim3(ET), smem, st, gt + (size_t)f0 * gfstride, r + (size_t)f0 * rfstride, rows,
                    cols, gpitch, gfstride, rpitch, rfstride, vec_ok, first_last + (size_t)f0 * 2, gbits,
                    partials + (size_t)f0 * nb * kKittiSums);
        DCMT_LAUNCH(k_kitti_finish, dim3((nf + 127) / 128), dim3(128), 0, st, partials + (size_t)f0 * nb * kKittiSums, nb, nf, out + f0);
    }
    return cudaGetLastError();
}

template cudaError_t kitti_run<float, float>(const float*, size_t, size_t, const float*, size_t, size_t, int, int, int, double*, int32_t*,
                                             unsigned*, KittiMetrics*, cudaStream_t);
template cudaError_t kitti_run<uint16_t, float>(const uint16_t*, size_t, size_t, const float*, size_t, size_t, int, int, int, double*,
                                                int32_t*, unsigned*, KittiMetrics*, cudaStream_t);
template cudaError_t kitti_run<uint16_t, uint16_t>(const uint16_t*, size_t, size_t, const uint16_t*, size_t, size_t, int, int, int,
                                                   double*, int32_t*, unsigned*, KittiMetrics*, cudaStream_t);

template <class G, class R>
cudaError_t eval_run(const G* gt, size_t gpitch, size_t gfstride, const R* r, size_t rpitch, size_t rfstride, int rows, int cols,
                     int n_frames, float tol, int mode, double* partials, EvalResult* out, cudaStream_t st) {
    const int nb = rows < kEvalMaxBlocks ? rows : kEvalMaxBlocks;
    const int vec_ok = vec4_ok(gt, gpitch, gfstride) && vec4_ok(r, rpitch, rfstride);
    for (int f0 = 0; f0 < n_frames; f0 += 65535) {  // gridDim.y limit
        const int nf = n_frames - f0 < 65535 ? n_frames - f0 : 65535;
        DCMT_LAUNCH((k_eval_partial<G, R>), dim3(nb, nf), dim3(ET), 0, st, gt + (size_t)f0 * gfstride, r + (size_t)f0 * rfstride, rows, cols,
                    gpitch, gfstride, rpitch, rfstride, tol, mode, vec_ok, partials + (size_t)f0 * nb * 4);
        DCMT_LAUNCH(k_eval_finish, dim3((nf + 127) / 128), dim3(128), 0, st, partials + (size_t)f0 * nb * 4, nb, nf, out + f0);
    }
    return cudaGetLastError();
}

template cudaError_t eval_run<float, float>(const float*, size_t, size_t, const float*, size_t, size_t, int, int, int, float, int,
                                            double*, EvalResult*, cudaStream_t);
template cudaError_t eval_run<uint16_t, float>(const uint16_t*, size_t, size_t, const float*, size_t, size_t, int, int, int, float, int,
                                               double*, EvalResult*, cudaStream_t);
template cudaError_t eval_run<uint16_t, uint16_t>(const uint16_t*, size_t, size_t, const uint16_t*, size_t, size_t, int, int, int, float,
                                                  int, double*, EvalResult*, cudaStream_t);

}  // namespace dcmt
