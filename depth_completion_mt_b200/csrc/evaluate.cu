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

}  // namespace

size_t eval_partial_doubles(int n_frames) { return (size_t)n_frames * kEvalMaxBlocks * 4; }

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
