// cuda_emu.h -- TEST INFRASTRUCTURE ONLY.  Minimal single-OS-thread CUDA execution-model emulator.
//
// Lets the *unmodified kernel sources* of depth_completion_mt_b200/csrc be compiled with g++
// (-DDCMT_EMU) and executed on the CPU, one thread block at a time, every CUDA thread a ucontext
// fiber that yields at barriers / warp collectives.  It exists so that `pytest -m "not gpu"` can
// diff the real kernel logic against the oracle in a container without a GPU.  It is never
// built into, loaded by or reachable from the product library (libdcmt.so) or the Python package;
// tests/emu/build_emu.py writes tests/emu/libdcmt_emu.so and only tests load it.
#pragma once
#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstddef>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <functional>

struct uint3 { unsigned x, y, z; };
struct dim3 {
    unsigned x, y, z;
    dim3(unsigned x_ = 1, unsigned y_ = 1, unsigned z_ = 1) : x(x_), y(y_), z(z_) {}
};
struct float2 { float x, y; };
struct alignas(16) float4 { float x, y, z, w; };
struct uint2 { unsigned x, y; };
struct int2 { int x, y; };
struct alignas(16) uint4 { unsigned x, y, z, w; };
struct alignas(16) int4 { int x, y, z, w; };
static inline int4 make_int4(int a, int b, int c, int d) { return int4{a, b, c, d}; }
struct ushort2 { unsigned short x, y; };
struct alignas(8) ushort4 { unsigned short x, y, z, w; };
static inline float4 make_float4(float a, float b, float c, float d) { return float4{a, b, c, d}; }
static inline float2 make_float2(float a, float b) { return float2{a, b}; }
static inline uint2 make_uint2(unsigned a, unsigned b) { return uint2{a, b}; }
static inline uint4 make_uint4(unsigned a, unsigned b, unsigned c, unsigned d) { return uint4{a, b, c, d}; }

typedef int cudaError_t;
enum { cudaSuccess = 0, cudaErrorInvalidValue = 1, cudaErrorMemoryAllocation = 2, cudaErrorNoDevice = 100 };
typedef void* cudaStream_t;
enum cudaMemcpyKind { cudaMemcpyHostToHost, cudaMemcpyHostToDevice, cudaMemcpyDeviceToHost, cudaMemcpyDeviceToDevice, cudaMemcpyDefault };
enum cudaFuncAttribute { cudaFuncAttributeMaxDynamicSharedMemorySize = 8 };

#define __global__
#define __device__
#define __host__
#define __forceinline__ inline __attribute__((always_inline))
#define __launch_bounds__(...)
#define __shared__ static
#define __align__(n) __attribute__((aligned(n)))
#define __grid_constant__

extern uint3 threadIdx, blockIdx;
extern dim3 blockDim, gridDim;

namespace dcmt_emu {
void launch(dim3 grid, dim3 block, size_t smem_bytes, const std::function<void()>& body);
void* dyn_smem();
void block_barrier();
int block_count(int pred);  // barrier + number of threads with pred != 0
unsigned warp_exchange(unsigned v, int width, int mode, int delta);  // shuffles inside segments of `width` lanes
unsigned warp_ballot(int pred);
unsigned warp_reduce_add(unsigned v);
int warp_gather(unsigned v, unsigned* out);  // all lanes' values; number of lanes in the warp
void warp_barrier();
long launches();
}  // namespace dcmt_emu

#define DCMT_DYN_SMEM(type, name) type* name = reinterpret_cast<type*>(dcmt_emu::dyn_smem())
namespace dcmt { void note_launch(); }
#define DCMT_LAUNCH(kernel, grid, block, smem, stream, ...) \
    (dcmt::note_launch(), dcmt_emu::launch((grid), (block), (smem), [=]() { kernel(__VA_ARGS__); }))

// ---- runtime shims (device memory == host memory) ----
static inline const char* cudaGetErrorString(cudaError_t e) { return e == cudaSuccess ? "no error" : "emulated CUDA error"; }
static inline cudaError_t cudaGetLastError() { return cudaSuccess; }
static inline cudaError_t cudaPeekAtLastError() { return cudaSuccess; }
static inline cudaError_t cudaGetDevice(int* d) { *d = 0; return cudaSuccess; }
static inline cudaError_t cudaGetDeviceCount(int* n) { *n = 1; return cudaSuccess; }
static inline cudaError_t cudaSetDevice(int d) { return d == 0 ? cudaSuccess : cudaErrorInvalidValue; }
static inline cudaError_t cudaMalloc(void** p, size_t n) { *p = std::malloc(n ? n : 1); if (*p) std::memset(*p, 0xCD, n); return *p ? cudaSuccess : cudaErrorMemoryAllocation; }
template <class T> static inline cudaError_t cudaMalloc(T** p, size_t n) { return cudaMalloc(reinterpret_cast<void**>(p), n); }
static inline cudaError_t cudaFree(void* p) { std::free(p); return cudaSuccess; }
static inline cudaError_t cudaMallocHost(void** p, size_t n) { *p = std::malloc(n ? n : 1); return *p ? cudaSuccess : cudaErrorMemoryAllocation; }
enum { cudaHostAllocDefault = 0, cudaHostAllocWriteCombined = 4 };
static inline cudaError_t cudaHostAlloc(void** p, size_t n, unsigned) { return cudaMallocHost(p, n); }
static inline cudaError_t cudaFreeHost(void* p) { std::free(p); return cudaSuccess; }
static inline cudaError_t cudaMemcpyAsync(void* d, const void* s, size_t n, cudaMemcpyKind, cudaStream_t = nullptr) { std::memcpy(d, s, n); return cudaSuccess; }
static inline cudaError_t cudaMemcpy(void* d, const void* s, size_t n, cudaMemcpyKind) { std::memcpy(d, s, n); return cudaSuccess; }
static inline cudaError_t cudaMemcpy2DAsync(void* d, size_t dp, const void* s, size_t sp, size_t w, size_t h, cudaMemcpyKind, cudaStream_t = nullptr) {
    for (size_t i = 0; i < h; ++i) std::memcpy((char*)d + i * dp, (const char*)s + i * sp, w);
    return cudaSuccess;
}
static inline cudaError_t cudaMemsetAsync(void* d, int v, size_t n, cudaStream_t = nullptr) { std::memset(d, v, n); return cudaSuccess; }
static inline cudaError_t cudaStreamSynchronize(cudaStream_t) { return cudaSuccess; }
enum { cudaStreamNonBlocking = 1 };
static inline cudaError_t cudaStreamCreateWithFlags(cudaStream_t* s, unsigned) { static char tok[8]; static int n = 0; *s = &tok[(n++) & 7]; return cudaSuccess; }
static inline cudaError_t cudaStreamDestroy(cudaStream_t) { return cudaSuccess; }
static inline cudaError_t cudaDeviceSynchronize() { return cudaSuccess; }
typedef int* cudaEvent_t;
static inline cudaError_t cudaEventCreate(cudaEvent_t* e) { *e = new int(0); return cudaSuccess; }
static inline cudaError_t cudaEventRecord(cudaEvent_t, cudaStream_t = nullptr) { return cudaSuccess; }
static inline cudaError_t cudaEventSynchronize(cudaEvent_t) { return cudaSuccess; }
static inline cudaError_t cudaEventElapsedTime(float* ms, cudaEvent_t, cudaEvent_t) { *ms = 0.f; return cudaSuccess; }
static inline cudaError_t cudaEventDestroy(cudaEvent_t e) { delete e; return cudaSuccess; }
template <class F> static inline cudaError_t cudaFuncSetAttribute(F, cudaFuncAttribute, int) { return cudaSuccess; }

// ---- device intrinsics ----
static inline void __syncthreads() { dcmt_emu::block_barrier(); }
static inline int __syncthreads_count(int p) { return dcmt_emu::block_count(p); }
static inline int __syncthreads_or(int p) { return dcmt_emu::block_count(p) != 0; }
static inline void __syncwarp(unsigned = 0xffffffffu) { dcmt_emu::warp_barrier(); }
template <class T> static inline T __ldg(const T* p) { return *p; }
template <class T> static inline T emu_shfl(T v, int mode, int arg, int width = 32) {
    static_assert(sizeof(T) == 4, "32-bit shuffles only");
    unsigned u; std::memcpy(&u, &v, 4);
    unsigned r = dcmt_emu::warp_exchange(u, width, mode, arg);
    T o; std::memcpy(&o, &r, 4); return o;
}
template <class T> static inline T __shfl_sync(unsigned, T v, int lane, int width = 32) { return emu_shfl(v, 0, lane, width); }
template <class T> static inline T __shfl_down_sync(unsigned, T v, int d, int width = 32) { return emu_shfl(v, 1, d, width); }
template <class T> static inline T __shfl_up_sync(unsigned, T v, int d, int width = 32) { return emu_shfl(v, 2, d, width); }
template <class T> static inline T __shfl_xor_sync(unsigned, T v, int m, int width = 32) { return emu_shfl(v, 3, m, width); }
// every lane of the warp makes the call, each with the mask of its own group (the __match_any_sync idiom)
static inline unsigned __reduce_add_sync(unsigned mask, unsigned v) {
    unsigned a[32], r = 0;
    const int n = dcmt_emu::warp_gather(v, a);
    for (int i = 0; i < n; ++i)
        if (mask >> i & 1u) r += a[i];
    return r;
}
static inline unsigned __match_any_sync(unsigned, unsigned v) {
    unsigned a[32], r = 0;
    const int n = dcmt_emu::warp_gather(v, a);
    for (int i = 0; i < n; ++i)
        if (a[i] == v) r |= 1u << i;
    return r;
}
static inline unsigned __ballot_sync(unsigned, int p) { return dcmt_emu::warp_ballot(p); }
static inline int __any_sync(unsigned, int p) { return dcmt_emu::warp_ballot(p) != 0; }
static inline int __all_sync(unsigned, int p) { return dcmt_emu::warp_ballot(!p) == 0; }
static inline long long clock64() { static long long c = 0; return ++c; }
static inline long long __double_as_longlong(double d) { long long u; std::memcpy(&u, &d, 8); return u; }
static inline double __longlong_as_double(long long u) { double d; std::memcpy(&d, &u, 8); return d; }
static inline unsigned __umulhi(unsigned a, unsigned b) { return (unsigned)(((unsigned long long)a * b) >> 32); }
static inline int __popc(unsigned v) { return __builtin_popcount(v); }
static inline int __clz(int v) { return v == 0 ? 32 : __builtin_clz((unsigned)v); }
static inline int __ffs(int v) { return __builtin_ffs(v); }
static inline unsigned __float_as_uint(float f) { unsigned u; std::memcpy(&u, &f, 4); return u; }
static inline float __uint_as_float(unsigned u) { float f; std::memcpy(&f, &u, 4); return f; }
static inline int __float_as_int(float f) { int u; std::memcpy(&u, &f, 4); return u; }
static inline float __int_as_float(int u) { float f; std::memcpy(&f, &u, 4); return f; }
static inline float __fadd_rn(float a, float b) { volatile float r = a + b; return r; }
static inline float __fsub_rn(float a, float b) { volatile float r = a - b; return r; }
static inline float __fmul_rn(float a, float b) { volatile float r = a * b; return r; }
static inline float __fdiv_rn(float a, float b) { volatile float r = a / b; return r; }
static inline double __dadd_rn(double a, double b) { volatile double r = a + b; return r; }
static inline double __dsub_rn(double a, double b) { volatile double r = a - b; return r; }
static inline double __dmul_rn(double a, double b) { volatile double r = a * b; return r; }
static inline double __ddiv_rn(double a, double b) { volatile double r = a / b; return r; }
static inline double __dsqrt_rn(double a) { volatile double r = std::sqrt(a); return r; }
static inline float __double2float_rn(double a) { return (float)a; }
static inline int __double2int_rz(double a) {
    if (a != a) return 0;
    if (a >= 2147483647.0) return 2147483647;
    if (a <= -2147483648.0) return (-2147483647 - 1);
    return (int)a;
}
static inline int __float2int_rz(float a) { return __double2int_rz((double)a); }
static inline float __int2float_rn(int a) { return (float)a; }
static inline unsigned __float2uint_rn(float a) { return (unsigned)std::nearbyintf(a); }
static inline float __uint2float_rn(unsigned a) { return (float)a; }
using std::max;
using std::min;
static inline int atomicAdd(int* p, int v) { int o = *p; *p += v; return o; }
static inline unsigned atomicAdd(unsigned* p, unsigned v) { unsigned o = *p; *p += v; return o; }
static inline int atomicMin(int* p, int v) { int o = *p; *p = std::min(o, v); return o; }
static inline int atomicMax(int* p, int v) { int o = *p; *p = std::max(o, v); return o; }
static inline unsigned atomicMin(unsigned* p, unsigned v) { unsigned o = *p; *p = std::min(o, v); return o; }
static inline unsigned atomicMax(unsigned* p, unsigned v) { unsigned o = *p; *p = std::max(o, v); return o; }
static inline unsigned long long atomicAdd(unsigned long long* p, unsigned long long v) { unsigned long long o = *p; *p += v; return o; }
static inline unsigned long long atomicMax(unsigned long long* p, unsigned long long v) { unsigned long long o = *p; *p = std::max(o, v); return o; }
static inline unsigned atomicCAS(unsigned* p, unsigned cmp, unsigned v) { unsigned o = *p; if (o == cmp) *p = v; return o; }
static inline int atomicOr(int* p, int v) { int o = *p; *p |= v; return o; }
static inline unsigned atomicOr(unsigned* p, unsigned v) { unsigned o = *p; *p |= v; return o; }
static inline int atomicExch(int* p, int v) { int o = *p; *p = v; return o; }
// packed 16-bit SIMD-in-word intrinsics
static inline unsigned emu_u16x2(unsigned a, unsigned b, bool is_max) {
    unsigned lo_a = a & 0xffffu, lo_b = b & 0xffffu, hi_a = a >> 16, hi_b = b >> 16;
    unsigned lo = is_max ? std::max(lo_a, lo_b) : std::min(lo_a, lo_b);
    unsigned hi = is_max ? std::max(hi_a, hi_b) : std::min(hi_a, hi_b);
    return lo | (hi << 16);
}
static inline unsigned __vmaxu2(unsigned a, unsigned b) { return emu_u16x2(a, b, true); }
static inline unsigned __vminu2(unsigned a, unsigned b) { return emu_u16x2(a, b, false); }
static inline unsigned __vadd2(unsigned a, unsigned b) { return ((a + b) & 0xffffu) | ((((a >> 16) + (b >> 16)) & 0xffffu) << 16); }
static inline unsigned __vsub2(unsigned a, unsigned b) { return ((a - b) & 0xffffu) | ((((a >> 16) - (b >> 16)) & 0xffffu) << 16); }
static inline unsigned __vimax3_u16x2(unsigned a, unsigned b, unsigned c) { return __vmaxu2(__vmaxu2(a, b), c); }
static inline unsigned __vimin3_u16x2(unsigned a, unsigned b, unsigned c) { return __vminu2(__vminu2(a, b), c); }
static inline unsigned __vcmpltu2(unsigned a, unsigned b) {
    return (((a & 0xffffu) < (b & 0xffffu)) ? 0xffffu : 0u) | (((a >> 16) < (b >> 16)) ? 0xffff0000u : 0u);
}
static inline unsigned __vcmpgeu2(unsigned a, unsigned b) { return ~__vcmpltu2(a, b); }
static inline unsigned __vcmpeq2(unsigned a, unsigned b) {
    return (((a & 0xffffu) == (b & 0xffffu)) ? 0xffffu : 0u) | (((a >> 16) == (b >> 16)) ? 0xffff0000u : 0u);
}
static inline unsigned __dp2a_lo(unsigned a, unsigned b, unsigned c) { return c + (a & 0xffffu) * (b & 0xffu) + (a >> 16) * ((b >> 8) & 0xffu); }
static inline unsigned __dp2a_hi(unsigned a, unsigned b, unsigned c) { return c + (a & 0xffffu) * ((b >> 16) & 0xffu) + (a >> 16) * (b >> 24); }
static inline unsigned __byte_perm(unsigned a, unsigned b, unsigned s) {
    unsigned long long v = ((unsigned long long)b << 32) | a;
    unsigned r = 0;
    for (int i = 0; i < 4; ++i) {
        unsigned sel = (s >> (4 * i)) & 0xf;
        unsigned byte = (unsigned)((v >> (8 * (sel & 7))) & 0xff);
        if (sel & 8) byte = (byte & 0x80) ? 0xff : 0x00;
        r |= byte << (8 * i);
    }
    return r;
}
static inline unsigned __funnelshift_r(unsigned lo, unsigned hi, unsigned s) {
    unsigned long long v = ((unsigned long long)hi << 32) | lo;
    return (unsigned)(v >> (s & 31));
}
static inline unsigned __funnelshift_l(unsigned lo, unsigned hi, unsigned s) {
    unsigned long long v = ((unsigned long long)hi << 32) | lo;
    return (unsigned)((v << (s & 31)) >> 32);
}
