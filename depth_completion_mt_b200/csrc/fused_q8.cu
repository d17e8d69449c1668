// fused_q8.cu -- the fast path of img_completion (/root/reference/src/DC_lidar_only/img_completion.cpp:17-204)
// for KITTI-style input: depth = uint16 / 256 (main.cpp:75-82), i.e. every pixel is 0 or k/256 with
// 26 <= k <= 25574 ("strict q8").  For such frames every stage up to and including the 5x5 Gaussian is exact
// integer arithmetic (SURVEY.md 0.4), so the whole pipeline runs on packed uint16x2 words:
//
//   encoding   e = 0                absent / -FLT_MAX (OpenCV's dilate border value)
//              e = q + 1            depth q/256 in inverted space;  hole <=> e == 1,  valid <=> e >= 27
//   k_q8_front   (A1..A4, :55-100)   invert, 2-tap dilate, close5, dilate7 + hole fill on a 2-D tile held in
//                                    shared memory; 7 passes fused, 128-bit shared-memory accesses, VIMNMX.U16x2 /
//                                    VIMNMX3.U16x2 / PRMT; writes a uint16 plane + per-column first/last keys
//   k_q8_tail    (A5..A10, :103-202) column extrapolation applied on load, 31x31 fill (vertical log-doubling +
//                                    ballot/popc-compacted horizontal pass over hole words only), median5 by
//                                    shared sorted columns + a 54-comparator selection network, Gaussian in
//                                    integer q16, final inversion, float32 store
//                                    holes that survive the first 31x31 fill (the reference's loop then runs more passes) are
//                                    resolved in the tile by a warp scanning growing squares of the A5 image in global memory
// Frames that are not strict q8 are detected (k_q8_classify or in-kernel validation) and go through generic.cu.
// No tensor cores: nothing here is a contraction.
#include "fused_q8.cuh"

#include <cstdlib>

#include "median_net.cuh"
#include "median_rows.cuh"
#include "rank_f32.cuh"

namespace dcmt {
namespace {

#ifndef DCMT_QT
#define DCMT_QT 256
#endif
#ifndef DCMT_QTT
#define DCMT_QTT 512
#endif
#ifndef DCMT_TAIL_CTAS
#define DCMT_TAIL_CTAS 2
#endif
#ifndef DCMT_FRONT_CTAS
#define DCMT_FRONT_CTAS 4
#endif
#ifndef DCMT_MEDIAN_ROWS
#define DCMT_MEDIAN_ROWS 1  // 1: shared-work median over runs of rows (median_rows.cuh); 0: independent selection networks
#endif
constexpr int QT = DCMT_QT;     // threads per CTA of k_q8_front (DCMT_FRONT_CTAS CTAs per SM on tiles of half the tail's height)
constexpr int QTT = DCMT_QTT;   // threads per CTA of k_q8_tail (2 CTAs per SM: their phases overlap)

#define SPLAT16(x) ((uint32_t)(x) | ((uint32_t)(x) << 16))
constexpr uint32_t E_VALID_MIN = 27;   // e >= 27  <=>  depth >= 0.1f  (26/256 = 0.1015625 is the smallest q8 value >= 0.1f)
constexpr uint32_t E_HUNDRED = 25601;  // encoding of 100.0 (empty-column fill, img_completion.cpp:110)
constexpr uint32_t kAbsMax = 0u;           // identity of max in the encoding (two lanes)

__device__ __forceinline__ uint32_t pmax(uint32_t a, uint32_t b) { return __vmaxu2(a, b); }
__device__ __forceinline__ uint32_t pmin(uint32_t a, uint32_t b) { return __vminu2(a, b); }
__device__ __forceinline__ uint32_t pmax3(uint32_t a, uint32_t b, uint32_t c) { return __vimax3_u16x2(a, b, c); }
__device__ __forceinline__ uint32_t pmin3(uint32_t a, uint32_t b, uint32_t c) { return __vimin3_u16x2(a, b, c); }
// (lo.hi16, hi.lo16): the pixel pair that starts one pixel to the right of `lo`
__device__ __forceinline__ uint32_t odd_pair(uint32_t lo, uint32_t hi) { return __byte_perm(lo, hi, 0x5432); }

template <bool kIsMax>
__device__ __forceinline__ uint32_t pext3(uint32_t a, uint32_t b, uint32_t c) {
    return kIsMax ? pmax3(a, b, c) : pmin3(a, b, c);
}
template <bool kIsMax>
__device__ __forceinline__ uint32_t pext(uint32_t a, uint32_t b) {
    return kIsMax ? pmax(a, b) : pmin(a, b);
}

__device__ __forceinline__ uint4 lds4(const uint32_t* p) { return *reinterpret_cast<const uint4*>(p); }
__device__ __forceinline__ void sts4(uint32_t* p, uint4 v) { *reinterpret_cast<uint4*>(p) = v; }
__device__ __forceinline__ uint2 lds2(const uint32_t* p) { return *reinterpret_cast<const uint2*>(p); }
__device__ __forceinline__ void sts2(uint32_t* p, uint2 v) { *reinterpret_cast<uint2*>(p) = v; }
__device__ __forceinline__ uint4 splat4(uint32_t v) { return make_uint4(v, v, v, v); }

// Iterates item = threadIdx.x, threadIdx.x + nt, ... over an (nr x nq) grid as (r, q) without a division: the
// descriptor (row length, per-step increments, magic reciprocal) is computed on the host for every row length a
// kernel uses; `lin` is the linear item index r * nq + q.
struct ItemsDesc {
    int nq, dr, dq, nt;
    uint32_t magic;  // floor(2^32 / nq) + 1
};
static ItemsDesc make_items(int nq, int nt) { return ItemsDesc{nq, nt / nq, nt % nq, nt, (uint32_t)((1ull << 32) / (unsigned)nq) + 1u}; }
struct Items {
    int r, q, lin, dr, dq, nq, nt;
    __device__ __forceinline__ explicit Items(const ItemsDesc& d) : dr(d.dr), dq(d.dq), nq(d.nq), nt(d.nt) {
        r = fast_div((int)threadIdx.x, d.magic);
        q = (int)threadIdx.x - r * d.nq;
        lin = threadIdx.x;
    }
    __device__ __forceinline__ void next() {
        q += dq;
        r += dr;
        lin += nt;
        if (q >= nq) { q -= nq; ++r; }
    }
};

// Encode one input pixel (metres, float) into inverted q8 (+1).  img_completion.cpp:55-67.
//   v = k/256, 26 <= k <= 25574  ->  e = 25601 - k  in [27, 25575]   (valid, inverted: 100 - v)
//   anything else a hole        ->  e = 1
// "Anything else" covers 0, negatives, values below 0.1f and values whose inversion 100 - v falls below 0.1f:
// all of them are holes for every later stage (each stage only asks `< 0.1f`, takes max/min with valid values
// or overwrites them), so their exact value never reaches the output.  What must hold for the integer pipeline to
// be exact is that every VALID pixel is a multiple of 1/256: kValidate checks it (the add of 2^23 must not round).
template <bool kValidate>
__device__ __forceinline__ uint32_t encode_bits(float v, float& bad) {
    const float t = fmaf(v, -256.0f, 25601.0f);  // 25601 - 256 v, exact for q8 input
    // valid <=> 26.5 <= t <= 25575.5 in ONE unsigned compare (positive floats order like their bit patterns; smaller,
    // negative and NaN t wrap to huge values).  For q8 input t is an integer, so this is exactly 27 <= t <= 25575,
    // i.e. 0.1f <= v and 0.1f <= 100 - v.  For other input the band is slightly wider than the reference's `>= 0.1f`
    // on purpose: every pixel the reference would treat as valid lands inside it with a non-integral t and trips
    // the validation, and everything outside it is a hole for the reference as well.
    const bool valid = __float_as_uint(t) - 0x41d40000u <= 0x46c7cf00u - 0x41d40000u;
    const float ef = valid ? t : 1.0f;
    const float m = ef + 8388608.0f;  // 2^23: the integer lands in the low mantissa bits
    if (kValidate) {
        // exact test that 256 v is the integer the encoding kept (t itself may round a near-grid value onto the grid, so
        // it cannot be used for this): K = 25601 - (m - 2^23); -K = m - (2^23 + 25601) is exact, and ONE FMA gives the
        // residual 256 v - K, which is zero iff v is on the grid
        const float res = fmaf(v, 256.0f, m - 8414209.0f);
        if (valid) bad = fmaf(res, res, bad);  // stays 0 iff every valid pixel seen so far is on the grid
    }
    return __float_as_uint(m);
}
template <bool kValidate>
__device__ __forceinline__ uint32_t encode_pair(float v0, float v1, float& bad) {
    return __byte_perm(encode_bits<kValidate>(v0, bad), encode_bits<kValidate>(v1, bad), 0x5410);
}

// thread -> (row r0, quad q) of a grid that is nq quads wide: q is fixed per thread, rows advance by nrt = QT / nq per
// sweep (threads with r0 >= nrt idle).  magic = floor(2^32 / nq) + 1 comes from the host: no division in the kernel.
struct ColMap {
    int nq, nrt;
    uint32_t magic;
};
static ColMap make_colmap(int nq, int nthreads) { return ColMap{nq, nthreads / nq, (uint32_t)((1ull << 32) / (unsigned)nq) + 1u}; }

struct FrontArgs {
    const float* in;              // float32 metres ...
    const uint16_t* in16;         // ... or KITTI uint16 (metres * 256), exactly one of the two
    size_t in_pitch, in_fstride;  // elements
    uint16_t* mid;                // rows x mid_pitch uint16 per frame
    size_t mid_pitch, mid_fstride;
    uint32_t* col_first;          // mid_pitch keys per frame: (row << 16) | e of the first valid row, atomicMin
    uint32_t* col_last;           // ... last valid row, atomicMax
    FrameCounters* ctr;
    int rows, cols, th, tw;
    int vec_ok;                   // input rows are 16-byte aligned: float4 loads
    int validate;                 // check strict q8-ness of every loaded pixel (DCMT_PATH_AUTO)
    ColMap m_load, m_pass, m_core;  // region (RQ quads), computed quads (RQ - 1), core quads (tw / 8)
    ItemsDesc i_half;               // half-quad columns of the computed quads: 2 (RQ - 1) per row of items
    long long* prof;              // optional: 16 clock64() stamps per CTA (debugging aid)
    int codes;                    // in16 holds CODES (the dictionary encoding of rank_f32.cu: already e), not KITTI uint16
    int use_tma;                  // k_q8_front: region loaded by one TMA box copy (else front_load's per-thread loads)
};

// ------------------------------------------------------------------------------------------------
// k_q8_front.  Region = core (th x tw) + {up 8, down 9} rows, {left 8, right 16} columns (the dependency cone is
// up 8 / down 9 / left 7 / right 9; widths are rounded to 8-pixel quads).  Two shared-memory planes; every pass reads
// neighbours from one with 128-bit loads and writes the other.
//
// Border handling costs nothing inside the passes:
//   * a thread owns one quad COLUMN for the whole kernel and walks down the rows, so "this quad is outside the image"
//     is a per-thread constant (such threads idle) and the in-image row range is a loop bound uniform over the CTA;
//   * cells outside the image are zeroed once in both planes and never written again, and every pass is a MAX:
//     the erosion half of close5 runs on complemented values (min(a, b) = ~max(~a, ~b)), so 0 is the identity the
//     next reader needs in every pass (absent tap, -FLT_MAX for the dilations, +FLT_MAX for the erosions);
//   * each pass computes exactly the rows / quads later passes need (the rest of the region holds stale values no
//     core pixel depends on), so nothing is clamped.
// A frame width that is not a multiple of 8 leaves one quad straddling the right edge: its outside lanes are masked
// in the kStraddle instantiation only.
// ------------------------------------------------------------------------------------------------
constexpr int FU = 8, FD = 9, FLQ = 1, FRQ = 2;  // rows up/down, quads left/right

#define DCMT_STAMP(a, k)                                                                                         \
    do {                                                                                                         \
        if ((a).prof && threadIdx.x == 0)                                                                        \
            (a).prof[((size_t)(blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x) * 16 + (k)] = clock64(); \
    } while (0)

struct Tile {
    int RH, RQ, pitchw;
    int rlo, rhi;  // region rows inside the image: [rlo, rhi)
    int qlo, qhi;  // region quads with at least one pixel inside the image: [qlo, qhi)
    int qs;        // the quad straddling the right image edge (cols % 8 != 0), or -1
    uint4 smask;   // its in-image lanes
};

__device__ __forceinline__ void tile_columns(Tile& t, int gx0, int cols) {
    t.qlo = gx0 < 0 ? (-gx0) / 8 : 0;  // gx0 is a multiple of 8
    t.qhi = min(t.RQ, (cols - gx0 + 7) / 8);
    t.qs = -1;
    t.smask = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);
    if (cols % 8 != 0) {
        const int q = (cols - gx0) / 8;
        if (q >= 0 && q < t.RQ) {
            t.qs = q;
            const int n = cols - (gx0 + q * 8);  // 1..7 pixels inside
            uint32_t m[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) m[j] = (2 * j < n ? 0x0000ffffu : 0u) | (2 * j + 1 < n ? 0xffff0000u : 0u);
            t.smask = make_uint4(m[0], m[1], m[2], m[3]);
        }
    }
}
__device__ __forceinline__ bool outside(const Tile& t, int r, int q) { return r < t.rlo || r >= t.rhi || q < t.qlo || q >= t.qhi; }
__device__ __forceinline__ uint4 blend(uint4 v, uint4 m, uint32_t ident) {
    return make_uint4((v.x & m.x) | (ident & ~m.x), (v.y & m.y) | (ident & ~m.y), (v.z & m.z) | (ident & ~m.z), (v.w & m.w) | (ident & ~m.w));
}
__device__ __forceinline__ uint4 and4(uint4 v, uint4 m) { return make_uint4(v.x & m.x, v.y & m.y, v.z & m.z, v.w & m.w); }

// what a thread needs to walk its quad column: first row, word offset of (r0, q), strides, activity, lane mask
struct ColThread {
    int r0, off0, nrt, dstep;
    bool act;     // the thread owns a quad with at least one pixel inside the image
    uint4 cmask;  // in-image lanes of that quad (all ones unless it straddles the right edge)
};
__device__ __forceinline__ ColThread col_thread(const ColMap& m, const Tile& t, int q_first) {
    ColThread c;
    c.r0 = fast_div((int)threadIdx.x, m.magic);
    const int q = (int)threadIdx.x - c.r0 * m.nq + q_first;
    c.off0 = (c.r0 * t.RQ + q) * 4;
    c.nrt = m.nrt;
    c.dstep = m.nrt * t.RQ * 4;
    c.act = c.r0 < m.nrt && q >= t.qlo && q < t.qhi;
    c.cmask = q == t.qs ? t.smask : make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);
    return c;
}

// One pass: rows [rb, re) of the thread's quad column, v = f(word offset).  rb <= 8 < nrt: at most one sweep is skipped.
template <bool kStraddle, class F>
__device__ __forceinline__ void col_pass(uint32_t* __restrict__ dst, const ColThread& c, int rb, int re, F f) {
    if (!c.act) return;
    int r = c.r0, off = c.off0;
    if (r < rb) { r += c.nrt; off += c.dstep; }
#pragma unroll 2
    for (; r < re; r += c.nrt, off += c.dstep) {
        uint4 v = f(off);
        if (kStraddle) v = and4(v, c.cmask);
        sts4(dst + off, v);
    }
}

template <int R, bool kIsMax>
__device__ __forceinline__ uint4 v_window(const uint32_t* __restrict__ p, int pitchw) {
    uint4 acc = lds4(p);
#pragma unroll
    for (int d = 1; d <= R; ++d) {
        const uint4 up = lds4(p - d * pitchw), dn = lds4(p + d * pitchw);
        acc.x = pext3<kIsMax>(acc.x, up.x, dn.x);
        acc.y = pext3<kIsMax>(acc.y, up.y, dn.y);
        acc.z = pext3<kIsMax>(acc.z, up.z, dn.z);
        acc.w = pext3<kIsMax>(acc.w, up.w, dn.w);
    }
    return acc;
}

// horizontal 5-window: out_j = ext(P_{j-1}, R_j, P_j, R_{j+1}, P_{j+1}),  R_j = (c_{2j-1}, c_{2j})
template <bool kIsMax>
__device__ __forceinline__ uint4 h5_window(const uint32_t* __restrict__ p) {
    const uint4 c = lds4(p);
    const uint32_t wl = p[-1], wr = p[4];
    const uint32_t r0 = odd_pair(wl, c.x), r1 = odd_pair(c.x, c.y), r2 = odd_pair(c.y, c.z), r3 = odd_pair(c.z, c.w),
                   r4 = odd_pair(c.w, wr);
    uint4 o;
    o.x = pext3<kIsMax>(pext3<kIsMax>(wl, r0, c.x), r1, c.y);
    o.y = pext3<kIsMax>(pext3<kIsMax>(c.x, r1, c.y), r2, c.z);
    o.z = pext3<kIsMax>(pext3<kIsMax>(c.y, r2, c.z), r3, c.w);
    o.w = pext3<kIsMax>(pext3<kIsMax>(c.z, r3, c.w), r4, wr);
    return o;
}

// horizontal 7-window max of one quad: out_j = max(R_{j-1}, R_j, R_{j+1}, R_{j+2}, P_{j-1}, P_j, P_{j+1})
__device__ __forceinline__ uint4 h7_max_quad(const uint32_t* __restrict__ p) {
    const uint4 c = lds4(p);
    const uint2 l = *reinterpret_cast<const uint2*>(p - 2);
    const uint2 rr = *reinterpret_cast<const uint2*>(p + 4);
    const uint32_t wm2 = l.x, wm1 = l.y, w0 = c.x, w1 = c.y, w2 = c.z, w3 = c.w, w4 = rr.x, w5 = rr.y;
    const uint32_t rm1 = odd_pair(wm2, wm1), r0 = odd_pair(wm1, w0), r1 = odd_pair(w0, w1), r2 = odd_pair(w1, w2),
                   r3 = odd_pair(w2, w3), r4 = odd_pair(w3, w4), r5 = odd_pair(w4, w5);
    uint4 o;
    o.x = pmax3(pmax3(rm1, r0, r1), pmax3(r2, wm1, w0), w1);
    o.y = pmax3(pmax3(r0, r1, r2), pmax3(r3, w0, w1), w2);
    o.z = pmax3(pmax3(r1, r2, r3), pmax3(r4, w1, w2), w3);
    o.w = pmax3(pmax3(r2, r3, r4), pmax3(r5, w2, w3), w4);
    return o;
}

// d = hole(d) ? t : d for two packed lanes, given t >= d >= 1 and holes == 1 exactly (img_completion.cpp:92-99):
//   a = d - 27 (mod 2^16) is huge for holes, small otherwise;  min(t - 27, a) + 27 picks t for holes, d otherwise.
__device__ __forceinline__ uint32_t fill_holes(uint32_t d, uint32_t t) {
    const uint32_t k = SPLAT16(65536 - 27);
    return __vadd2(pmin(__vadd2(t, k), __vadd2(d, k)), SPLAT16(27));
}

// ---- vertical passes: one item = one half-quad column (2 words, 4 pixels) x a run of L consecutive rows.  The rows
// a window needs are loaded once and slide through registers, so a 5-row window costs (L + 4) / L loads per output
// instead of 5 -- the front kernel is bound by shared-memory bandwidth, not by instruction issue.
__device__ __forceinline__ uint2 half_mask(const Tile& t, int h) {
    if ((h >> 1) != t.qs) return make_uint2(0xffffffffu, 0xffffffffu);
    return (h & 1) ? make_uint2(t.smask.z, t.smask.w) : make_uint2(t.smask.x, t.smask.y);
}

// dst(r) = max of src over rows r-2 .. r+2, rows [rb, re)
template <bool kStraddle, int L>
__device__ __forceinline__ void v5max_runs(const uint32_t* __restrict__ src, uint32_t* __restrict__ dst, const Tile& t, const ItemsDesc& d,
                                           int rb, int re) {
    const int pw = t.pitchw, nseg = (re - rb + L - 1) / L;
    for (Items i(d); i.r < nseg; i.next()) {
        const int h = i.q, q = h >> 1;
        if (q < t.qlo || q >= t.qhi) continue;
        const int rf = rb + i.r * L, n = min(L, re - rf);
        const uint32_t* p = src + (rf - 2) * pw + 2 * h;
        uint32_t* o = dst + rf * pw + 2 * h;
        const uint2 m = half_mask(t, h);
        uint2 w0 = lds2(p), w1 = lds2(p + pw), w2 = lds2(p + 2 * pw), w3 = lds2(p + 3 * pw);
        auto step = [&](int k) {
            const uint2 w4 = lds2(p + (k + 4) * pw);
            uint2 v = make_uint2(pmax3(pmax3(w0.x, w1.x, w2.x), w3.x, w4.x), pmax3(pmax3(w0.y, w1.y, w2.y), w3.y, w4.y));
            if (kStraddle) { v.x &= m.x; v.y &= m.y; }
            sts2(o + k * pw, v);
            w0 = w1; w1 = w2; w2 = w3; w3 = w4;
        };
        if (n == L) {  // full run: no guards
#pragma unroll
            for (int k = 0; k < L; ++k) step(k);
        } else {
#pragma unroll
            for (int k = 0; k < L; ++k)
                if (k < n) step(k);
        }
    }
}

// The vertical erosion of close5 and the vertical half of dilate7 in one sweep (:85, :88-90), for core rows [rb, re):
//   D(r)  = ~max(Y'(r-2 .. r+2))   Y' = complemented horizontal erosion; rows outside the image give D = 0 (absent)
//   V7(r) =  max(D(r-3 .. r+3))
// D goes to the core-sized plane C (core quads only: pass 7 reads nothing else of it), V7 to plane V.
template <bool kStraddle, int L>
__device__ __forceinline__ void v_close_dilate_runs(const uint32_t* __restrict__ Y, uint32_t* __restrict__ V, uint32_t* __restrict__ C,
                                                    const Tile& t, const ItemsDesc& d, int rb, int re, int cq) {
    const int pw = t.pitchw, cpw = cq * 4, nseg = (re - rb + L - 1) / L;
    for (Items i(d); i.r < nseg; i.next()) {
        const int h = i.q, q = h >> 1;
        if (q < t.qlo || q >= t.qhi) continue;
        const int rf = rb + i.r * L, n = min(L, re - rf);
        const uint32_t* p = Y + (rf - 5) * pw + 2 * h;
        uint32_t* ov = V + rf * pw + 2 * h;
        const bool core = q >= FLQ && q < FLQ + cq;
        uint32_t* od = C + (rf - FU) * cpw + (2 * h - FLQ * 4);
        const uint2 m = half_mask(t, h);
        uint2 y0 = lds2(p), y1 = lds2(p + pw), y2 = lds2(p + 2 * pw), y3 = lds2(p + 3 * pw);
        uint2 dw[7];
        auto step = [&](int e, bool check_rows) {  // D row rf - 3 + e, V7 row rf + e - 6
            const uint2 y4 = lds2(p + (e + 4) * pw);
            uint2 dn = make_uint2(~pmax3(pmax3(y0.x, y1.x, y2.x), y3.x, y4.x), ~pmax3(pmax3(y0.y, y1.y, y2.y), y3.y, y4.y));
            if (kStraddle) { dn.x &= m.x; dn.y &= m.y; }
            if (check_rows) {
                const int row = rf - 3 + e;
                if (row < t.rlo || row >= t.rhi) dn = make_uint2(0u, 0u);
            }
            y0 = y1; y1 = y2; y2 = y3; y3 = y4;
            dw[e % 7] = dn;
            if (e >= 3 && e < 3 + L && e - 3 < n && core) sts2(od + (e - 3) * cpw, dn);
            if (e >= 6) {
                const uint2 v = make_uint2(pmax3(pmax3(dw[0].x, dw[1].x, dw[2].x), pmax3(dw[3].x, dw[4].x, dw[5].x), dw[6].x),
                                           pmax3(pmax3(dw[0].y, dw[1].y, dw[2].y), pmax3(dw[3].y, dw[4].y, dw[5].y), dw[6].y));
                sts2(ov + (e - 6) * pw, v);
            }
        };
        if (n == L && rf - 3 >= t.rlo && rf + L + 3 <= t.rhi) {  // full run, every D row inside the image: no guards
#pragma unroll
            for (int e = 0; e < L + 6; ++e) step(e, false);
        } else {
#pragma unroll
            for (int e = 0; e < L + 6; ++e)
                if (e < n + 6) step(e, true);
        }
    }
}

// The two horizontal passes of close5 (:84-85) on one quad in registers: dilate5 on words -1 .. 4, complement (0 where
// the word lies outside the image: absent for the erosion), erode5 as a max of complements on words 0 .. 3.  The result
// stays complemented (Y') for the vertical erosion.  ml / mr: in-image lanes of words -1 / 4, mc: of the quad itself.
__device__ __forceinline__ uint4 h5_close_quad(const uint32_t* __restrict__ p, uint32_t ml, uint4 mc, uint32_t mr) {
    const uint2 l = lds2(p - 2), r = lds2(p + 4);
    const uint4 c = lds4(p);
    const uint32_t P[8] = {l.x, l.y, c.x, c.y, c.z, c.w, r.x, r.y};  // P[j + 2] = word j
    uint32_t R[7];                                                     // R[j + 1] = odd pair (word j-1, word j), j = -1 .. 5
#pragma unroll
    for (int j = 0; j < 7; ++j) R[j] = odd_pair(P[j], P[j + 1]);
    uint32_t m[6];  // m[j + 1] = dilate5 at word j, j = -1 .. 4
#pragma unroll
    for (int j = 0; j < 6; ++j) m[j] = pmax3(pmax3(P[j], R[j], P[j + 1]), R[j + 1], P[j + 2]);
    m[0] = ~m[0] & ml;
    m[1] = ~m[1] & mc.x;
    m[2] = ~m[2] & mc.y;
    m[3] = ~m[3] & mc.z;
    m[4] = ~m[4] & mc.w;
    m[5] = ~m[5] & mr;
    uint32_t S[5];  // S[j] = odd pair (m word j-1, m word j), j = 0 .. 4
#pragma unroll
    for (int j = 0; j < 5; ++j) S[j] = odd_pair(m[j], m[j + 1]);
    uint4 o;
    o.x = pmax3(pmax3(m[0], S[0], m[1]), S[1], m[2]);
    o.y = pmax3(pmax3(m[1], S[1], m[2]), S[2], m[3]);
    o.z = pmax3(pmax3(m[2], S[2], m[3]), S[3], m[4]);
    o.w = pmax3(pmax3(m[3], S[3], m[4]), S[4], m[5]);
    return o;
}

// Passes 1-6 on region rows (core rows are [FU, FU + th)); each pass covers the rows the later ones read:
//   pass 7 needs V7 on the core rows <- D on core +- 3 <- H5 on core +- 5 (<- V5max on the same rows) <- 2-tap on core +- 7.
// Four trips through shared memory: 2-tap, V5max (vertical runs), H5max + H5min (fused per quad), V5min + V7max (fused
// vertical runs).
template <bool kStraddle>
__device__ __forceinline__ void front_passes(uint32_t* A, uint32_t* B, uint32_t* C, const Tile& t, const ColThread& c, const ItemsDesc& halves,
                                             int th, int cq) {
    const int pw = t.pitchw;
    auto rb = [&](int lo) { return max(lo, t.rlo); };
    auto re = [&](int hi) { return min(hi, t.rhi); };
    // ---- pass 1: 2-tap dilate (:71-80)  out(y,x) = max(in(y-1,x+1), in(y+2,x+2)), absent taps = -FLT_MAX (e = 0)
    col_pass<kStraddle>(B, c, rb(FU - 7), re(FU + th + 7), [&](int off) {
        const uint32_t* pa = A + off - pw;      // row y-1
        const uint32_t* pb = A + off + 2 * pw;  // row y+2
        const uint4 ca = lds4(pa), cb = lds4(pb);
        const uint32_t na = pa[4], nb = pb[4];
        // tap 1: pixels (x+1, x+2) of row y-1; tap 2: pixels (x+2, x+3) of row y+2
        return make_uint4(pmax(odd_pair(ca.x, ca.y), cb.y), pmax(odd_pair(ca.y, ca.z), cb.z), pmax(odd_pair(ca.z, ca.w), cb.w),
                          pmax(odd_pair(ca.w, na), nb));
    });
    __syncthreads();
    // ---- pass 2: vertical half of dilate5 (:84)
    v5max_runs<kStraddle, 9>(B, A, t, halves, rb(FU - 5), re(FU + th + 5));
    __syncthreads();
    // ---- passes 3 + 4: horizontal dilate5 and horizontal erode5, fused per quad; output complemented
    {
        const int q = (c.off0 >> 2) - c.r0 * t.RQ;  // the thread's quad column
        const uint32_t ml = (q - 1 >= t.qlo && q - 1 < t.qhi) ? (q - 1 == t.qs ? t.smask.w : 0xffffffffu) : 0u;
        const uint32_t mr = (q + 1 >= t.qlo && q + 1 < t.qhi) ? (q + 1 == t.qs ? t.smask.x : 0xffffffffu) : 0u;
        col_pass<kStraddle>(B, c, rb(FU - 5), re(FU + th + 5), [&](int off) { return h5_close_quad(A + off, ml, c.cmask, mr); });
    }
    __syncthreads();
    // ---- passes 5 + 6: vertical erode5 -> D (plane C, core quads) and vertical half of dilate7 (:88-90) -> A
    v_close_dilate_runs<kStraddle, 8>(B, A, C, t, halves, rb(FU), re(FU + th), cq);
    __syncthreads();
}

// Encode two KITTI uint16 pixels (k = metres * 256, main.cpp:75-82) packed in one word: the convertTo(CV_32F, 1/256)
// of main.cpp:79 and the inversion of img_completion.cpp:55-67 in integer form.  Per lane: t = 25601 - k (mod 2^16);
// the pixel is valid iff 27 <= t <= 25575 (<=> 26 <= k <= 25574), otherwise it is a hole (e = 1).
__device__ __forceinline__ uint32_t encode_u16_pair(uint32_t w) {
    const uint32_t t = __vsub2(SPLAT16(25601), w);
    const uint32_t u = __vsub2(t, SPLAT16(27));              // valid lanes: 0 .. 25548
    const uint32_t c = pmin(u, SPLAT16(25549)) ^ SPLAT16(25549);  // zero lane <=> invalid; both operands < 0x8000
    const uint32_t nz = ((c + SPLAT16(0x7fff)) >> 15) & 0x00010001u;  // 1 per valid lane (no carry between lanes)
    const uint32_t m = nz * 0xffffu;                          // 0xffff per valid lane
    return (t & m) | (SPLAT16(1) & ~m);
}

// pass 0: load, validate, invert, encode (:55-67) into plane A; cells outside the image are zeroed in BOTH planes.
// Sweeps go in batches of three so that up to six 16-byte global loads per thread are in flight before the first
// one is consumed.  kIn16: KITTI uint16 input (one 16-byte load per quad, no validation needed).
template <bool kIn16, bool kValidate, bool kCodes = false>
__device__ __forceinline__ void front_load(const FrontArgs& a, const void* in0v, uint32_t* A, uint32_t* B, const Tile& t, int gx0,
                                           float& bad) {
    // in0 points at region cell (0, 0) of the frame (possibly outside the buffer: only in-image cells are read)
    const float* in0 = static_cast<const float*>(in0v);
    const uint16_t* in0h = static_cast<const uint16_t*>(in0v);
    const ColMap& m = a.m_load;
    const int r0 = fast_div((int)threadIdx.x, m.magic), q = (int)threadIdx.x - r0 * m.nq;
    if (r0 >= m.nrt) return;
    const int pitch = (int)a.in_pitch, gx = gx0 + q * 8;
    const bool q_in = q >= t.qlo && q < t.qhi;
    const bool vec = q_in && q != t.qs && a.vec_ok;
    const int dstep = m.nrt * t.pitchw;
    int r = r0, off = (r0 * t.RQ + q) * 4;
#pragma unroll 1
    while (r < t.RH) {
        float4 f0[3], f1[3];
        uint4 h[3];
        int offs[3], rr[3];
        bool live[3], in[3];
#pragma unroll
        for (int u = 0; u < 3; ++u) {
            offs[u] = off;
            rr[u] = r;
            live[u] = r < t.RH;
            in[u] = live[u] && q_in && r >= t.rlo && r < t.rhi;
            f0[u] = f1[u] = make_float4(0.f, 0.f, 0.f, 0.f);
            h[u] = make_uint4(0u, 0u, 0u, 0u);
            if (in[u] && vec) {
                if (kIn16) {
                    h[u] = __ldg(reinterpret_cast<const uint4*>(in0h + (r * pitch + q * 8)));
                } else {
                    const float4* p = reinterpret_cast<const float4*>(in0 + (r * pitch + q * 8));
                    f0[u] = __ldg(p);
                    f1[u] = __ldg(p + 1);
                }
            }
            r += m.nrt;
            off += dstep;
        }
#pragma unroll
        for (int u = 0; u < 3; ++u) {
            if (!live[u]) continue;
            if (!in[u]) {  // outside the image: absent, in both planes, for good
                sts4(A + offs[u], splat4(0u));
                sts4(B + offs[u], splat4(0u));
                continue;
            }
            uint4 o;
            if (vec) {
                if (kCodes) {
                    o = h[u];
                } else if (kIn16) {
                    o = make_uint4(encode_u16_pair(h[u].x), encode_u16_pair(h[u].y), encode_u16_pair(h[u].z), encode_u16_pair(h[u].w));
                } else {
                    o.x = encode_pair<kValidate>(f0[u].x, f0[u].y, bad);
                    o.y = encode_pair<kValidate>(f0[u].z, f0[u].w, bad);
                    o.z = encode_pair<kValidate>(f1[u].x, f1[u].y, bad);
                    o.w = encode_pair<kValidate>(f1[u].z, f1[u].w, bad);
                }
            } else {  // unaligned rows or the quad straddling the right edge: scalar loads, outside lanes absent
                uint32_t e[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    e[j] = 0u;
                    if (gx + j < a.cols) {
                        if (kCodes) e[j] = (uint32_t)__ldg(in0h + (rr[u] * pitch + q * 8 + j));
                        else if (kIn16) e[j] = encode_u16_pair((uint32_t)__ldg(in0h + (rr[u] * pitch + q * 8 + j))) & 0xffffu;
                        else e[j] = encode_bits<kValidate>(__ldg(in0 + (rr[u] * pitch + q * 8 + j)), bad) & 0xffffu;
                    }
                }
                o = make_uint4(e[0] | (e[1] << 16), e[2] | (e[3] << 16), e[4] | (e[5] << 16), e[6] | (e[7] << 16));
            }
            sts4(A + offs[u], o);
        }
    }
}

// pass 0 from a region staged in shared memory by one TMA box copy: RH rows x RQ * 8 pixels at S (row r of the box at
// word r * RQ * 8 for float input, r * RQ * 4 for uint16), zero wherever the box leaves the image.  The staged floats
// fill planes A and B, so every thread first decodes its quads into registers -- at most kStagedSweeps per thread, the
// host uses front_load beyond that -- and writes A only after the barrier.  Cells outside the image are decided by
// position, as in front_load, and zeroed in both planes: the zero fill itself would encode as a hole, not as absent.
constexpr int kStagedSweeps = 6;
template <bool kIn16, bool kValidate, bool kCodes = false>
__device__ __forceinline__ void front_decode_staged(const FrontArgs& a, const uint32_t* S, uint32_t* A, uint32_t* B, const Tile& t,
                                                    float& bad) {
    const ColMap& m = a.m_load;
    const int r0 = fast_div((int)threadIdx.x, m.magic), q = (int)threadIdx.x - r0 * m.nq;
    const bool q_in = r0 < m.nrt && q >= t.qlo && q < t.qhi;
    const int sstep = m.nrt * (kIn16 ? t.pitchw : 2 * t.pitchw);
    const uint32_t* p = S + r0 * (kIn16 ? t.pitchw : 2 * t.pitchw) + q * (kIn16 ? 4 : 8);
    uint4 o[kStagedSweeps];
#pragma unroll
    for (int u = 0; u < kStagedSweeps; ++u, p += sstep) {
        const int r = r0 + u * m.nrt;
        o[u] = splat4(0u);
        if (!q_in || r < t.rlo || r >= t.rhi) continue;
        if (kCodes) {
            o[u] = lds4(p);
        } else if (kIn16) {
            const uint4 h = lds4(p);
            o[u] = make_uint4(encode_u16_pair(h.x), encode_u16_pair(h.y), encode_u16_pair(h.z), encode_u16_pair(h.w));
        } else {
            const uint4 f0 = lds4(p), f1 = lds4(p + 4);
            o[u] = make_uint4(encode_pair<kValidate>(__uint_as_float(f0.x), __uint_as_float(f0.y), bad),
                              encode_pair<kValidate>(__uint_as_float(f0.z), __uint_as_float(f0.w), bad),
                              encode_pair<kValidate>(__uint_as_float(f1.x), __uint_as_float(f1.y), bad),
                              encode_pair<kValidate>(__uint_as_float(f1.z), __uint_as_float(f1.w), bad));
        }
        if (q == t.qs) o[u] = and4(o[u], t.smask);  // lanes right of the image: absent
    }
    __syncthreads();  // every staged value is in registers: A and B may be overwritten
    if (r0 >= m.nrt) return;
    int off = (r0 * t.RQ + q) * 4;
#pragma unroll
    for (int u = 0; u < kStagedSweeps; ++u, off += m.nrt * t.pitchw) {
        const int r = r0 + u * m.nrt;
        if (r >= t.RH) break;
        sts4(A + off, o[u]);
        if (!q_in || r < t.rlo || r >= t.rhi) sts4(B + off, splat4(0u));
    }
}

template <bool kStraddle>
__global__ void __launch_bounds__(QT, DCMT_FRONT_CTAS) k_q8_front(FrontArgs a, const __grid_constant__ TensorMap3D tmap) {
    DCMT_DYN_SMEM(uint32_t, smem);
    __shared__ __align__(8) uint64_t s_bar;  // mbarrier the TMA tile load signals
    const int th = a.th, tw = a.tw, rows = a.rows, cols = a.cols;
    Tile t;
    t.RH = th + FU + FD;
    t.RQ = tw / 8 + FLQ + FRQ;
    t.pitchw = t.RQ * 4;
    // one quad of padding in front of plane A and behind plane B: the horizontal passes read one word beyond the
    // ends of a row (values no needed cell depends on, but the addresses must exist)
    uint32_t* A = smem + 4;
    uint32_t* B = A + t.RH * t.pitchw;
    uint32_t* C = B + t.RH * t.pitchw + 4;  // D = close5 result on the core: th rows x tw / 8 quads
    const int frame = blockIdx.z;  // slot == frame offset inside the chunk
    const int y0 = blockIdx.y * th, x0 = blockIdx.x * tw;
    const int gy0 = y0 - FU;
    const int gx0 = x0 - FLQ * 8;
    t.rlo = max(0, -gy0);
    t.rhi = min(t.RH, rows - gy0);
    tile_columns(t, gx0, cols);
    const ptrdiff_t origin = (ptrdiff_t)frame * (ptrdiff_t)a.in_fstride + ((ptrdiff_t)gy0 * (ptrdiff_t)a.in_pitch + gx0);

    DCMT_STAMP(a, 0);
    float bad = 0.0f;
    if (a.use_tma) {
        // ONE box copy of the region (zero outside the image) to the start of the dynamic shared memory, which is 128-byte
        // aligned: RH x RQ * 8 floats fill A and B exactly (A starts one quad in, B ends one quad short of the allocation)
        if (threadIdx.x == 0) {
            tma_bar_init(&s_bar);
            tma_load_3d(smem, &tmap, gx0, gy0, frame, &s_bar, (uint32_t)(t.RH * t.pitchw * (a.in16 ? 4 : 8)));
        }
        __syncthreads();  // the mbarrier is initialised before anyone waits on it
        tma_bar_wait(&s_bar, 0);
        if (a.in16 && a.codes) front_decode_staged<true, false, true>(a, smem, A, B, t, bad);
        else if (a.in16) front_decode_staged<true, false>(a, smem, A, B, t, bad);
        else if (a.validate) front_decode_staged<false, true>(a, smem, A, B, t, bad);
        else front_decode_staged<false, false>(a, smem, A, B, t, bad);
    } else if (a.in16 && a.codes) front_load<true, false, true>(a, a.in16 + origin, A, B, t, gx0, bad);  // dictionary codes (rank_f32.cu)
    else if (a.in16) front_load<true, false>(a, a.in16 + origin, A, B, t, gx0, bad);  // uint16 input is q8 by construction
    else if (a.validate) front_load<false, true>(a, a.in + origin, A, B, t, gx0, bad);
    else front_load<false, false>(a, a.in + origin, A, B, t, gx0, bad);
    if (__syncthreads_or(bad != 0.0f)) {  // not strict q8: this frame is redone by the generic pipeline
        if (threadIdx.x == 0) a.ctr[frame].needs_generic = 1;
        return;
    }
    DCMT_STAMP(a, 1);
    const ColThread c = col_thread(a.m_pass, t, 0);  // quads 0 .. RQ-2: the last halo quad is only ever read
    front_passes<kStraddle>(A, B, C, t, c, a.i_half, th, tw / 8);
    DCMT_STAMP(a, 2);

    // ---- pass 7: horizontal half of dilate7, hole fill (:92-100), store the core
    uint16_t* mid = a.mid + (size_t)frame * a.mid_fstride;
    {
        const ColMap& m = a.m_core;
        const int r0 = fast_div((int)threadIdx.x, m.magic), q = (int)threadIdx.x - r0 * m.nq;
        const int gx = x0 + q * 8;
        const int rend = min(th, rows - y0);
        if (r0 < m.nrt && gx < cols) {
            const int dstep = m.nrt * t.pitchw;
            int off = ((r0 + FU) * t.RQ + q + FLQ) * 4;
            const int cstep = m.nrt * m.nq * 4;
            uint32_t* pc = C + (r0 * m.nq + q) * 4;
            uint16_t* mp = mid + (size_t)(y0 + r0) * a.mid_pitch + gx;
            const size_t mstep = (size_t)m.nrt * a.mid_pitch;
#pragma unroll 2
            for (int r = r0; r < rend; r += m.nrt, off += dstep, pc += cstep, mp += mstep) {
                const uint4 tt = h7_max_quad(A + off);
                uint4 d = lds4(pc);
                d.x = fill_holes(d.x, tt.x);
                d.y = fill_holes(d.y, tt.y);
                d.z = fill_holes(d.z, tt.z);
                d.w = fill_holes(d.w, tt.w);
                sts4(pc, d);  // only this thread touches this quad of C in this pass
                *reinterpret_cast<uint4*>(mp) = d;
            }
        }
    }
    __syncthreads();
    DCMT_STAMP(a, 3);
    // ---- per-column first / last valid row inside this tile (feeds :103-129), merged across tiles by atomics.
    //      Two threads per column: one searches from the top, one from the bottom.
    const uint16_t* Ch = reinterpret_cast<const uint16_t*>(C);
    const int hrows = min(th, rows - y0);
    for (int c2 = threadIdx.x; c2 < 2 * tw; c2 += QT) {
        const int col = c2 >> 1, from_bottom = c2 & 1;
        const int gx = x0 + col;
        if (gx >= cols) continue;
        const uint16_t* p = Ch + col;
        if (!from_bottom) {
            for (int cy = 0; cy < hrows; ++cy) {
                const uint32_t e = p[(size_t)cy * tw];
                if (e >= E_VALID_MIN) {
                    atomicMin(a.col_first + (size_t)frame * a.mid_pitch + gx, ((uint32_t)(y0 + cy) << 16) | e);
                    break;
                }
            }
        } else {
            for (int cy = hrows - 1; cy >= 0; --cy) {
                const uint32_t e = p[(size_t)cy * tw];
                if (e >= E_VALID_MIN) {
                    atomicMax(a.col_last + (size_t)frame * a.mid_pitch + gx, ((uint32_t)(y0 + cy) << 16) | e);
                    break;
                }
            }
        }
    }
    DCMT_STAMP(a, 4);
}

// ------------------------------------------------------------------------------------------------
// k_q8_guided_front: the front of interpolate_with_superpixels (src/DC_lidar_camera/img_completion_lc.cpp:34-145) for
// strict-q8 input.  The reference runs, for every superpixel c, a 2-tap dilate and a 5x5 close on a copy of the image in
// which every pixel of another superpixel is 0 (:78-103), and keeps the result inside c.  Per output pixel p with label
// c (SURVEY.md App. B):
//     M_c(s)  = label(s) == c ? D(s) : 0                    (absent outside the image)
//     R1_c(r) = max(M_c(r + (-1,+1)), M_c(r + (+2,+2)))      r inside the image
//     R2_c(q) = max over r in 5x5(q), r inside the image, of R1_c(r)
//     out(p)  = min over q in 5x5(p), q inside the image, of R2_c(q);          out(p) = D(p) if p has no valid label.
// One thread computes one packed word = two horizontally adjacent pixels, each lane with its own label: the 12 x 10
// footprint is masked row by row (3 ALU ops per word: packed compare, min with 1, select), and because
//     max over a 5-window of R1 = max(5-window max of the tap-1 row, 5-window max of the tap-2 row three rows further down)
// every masked row contributes just six sliding 5-wide maxima; the vertical dilation runs over a ring of five such rows,
// the erosion over the five results.  About 430 lane-operations per pixel; the generic float kernel needs 3 600.
// Hole-class values are interchangeable (every later stage only asks `< 0.1`), so other-label pixels and holes both
// encode as 1.  Afterwards the kernel continues like k_q8_front: vertical / horizontal dilate7, hole fill, uint16 store,
// column keys -- and k_q8_tail finishes the frame.
// ------------------------------------------------------------------------------------------------
#ifndef DCMT_GTL
#define DCMT_GTL 512
#endif
#ifndef DCMT_GUIDED_CTAS
#define DCMT_GUIDED_CTAS 2
#endif
constexpr int GTL = DCMT_GTL;  // per-label kernel: DCMT_GUIDED_CTAS CTAs per SM, every warp works on one (or two) superpixels at a time
constexpr int GTW = 256;   // word-by-word kernel: two CTAs per SM, up to 128 registers per thread

struct GuidedArgs {
    FrontArgs f;            // geometry, input, outputs (column maps built for GT threads)
    const int32_t* labels;  // rows x cols int32 per frame, contiguous
    int n_clusters;
    int per_label;          // 1: one warp per superpixel (guided_label_warp); 0: every word on its own (guided_word)
    int* tile_flags;        // per tile: set by the per-label kernel when the tile is left to the word-by-word kernel
};

// lanes of `w` that lie inside the image -> 0xffff, given the image column of the low lane
__device__ __forceinline__ uint32_t lanes_inside(int gx, int cols) {
    return ((gx >= 0 && gx < cols) ? 0x0000ffffu : 0u) | ((gx + 1 >= 0 && gx + 1 < cols) ? 0xffff0000u : 0u);
}

template <bool kBorder>
__device__ __forceinline__ uint32_t guided_word(const uint32_t* __restrict__ A, const uint32_t* __restrict__ LB, int pitchw, int r, int w,
                                                uint32_t C, int gy, int gx, int rows, int cols) {
    // masked footprint rows k = 0 .. 11 <-> image rows gy - 5 + k; positions idx = 0 .. 9 <-> lane-0 columns gx - 3 + idx
    uint32_t cm[9];  // kBorder: in-image lanes of the R1 columns jj = 0 .. 8 (lane-0 column gx - 4 + jj)
    if (kBorder) {
#pragma unroll
        for (int jj = 0; jj < 9; ++jj) cm[jj] = lanes_inside(gx - 4 + jj, cols);
    }
    uint32_t ha[3][5];    // 5-window maxima of the tap-1 rows, waiting three rows for their tap-2 partner
    uint32_t ring[5][5];  // H rows (horizontal dilation of R1) for the vertical dilation
    uint32_t out = 0xffffffffu;
#pragma unroll
    for (int k = 0; k < 12; ++k) {
        const uint32_t* pa = A + (r - 5 + k) * pitchw + (w - 2);
        const uint32_t* pl = LB + (r - 5 + k) * pitchw + (w - 2);
        uint32_t d[6], l[6];
#pragma unroll
        for (int u = 0; u < 6; ++u) { d[u] = pa[u]; l[u] = pl[u]; }
        // masked value: same label -> the pixel itself; other label -> 0, i.e. a hole (e = 1); outside the image ->
        // absent (0 stays 0).  ne = 1 per lane whose label differs; cap = 0xffff - 0xfffe * ne (one IMAD, lanes cannot
        // borrow); masked = min(value, cap).
        uint32_t m[10];
#pragma unroll
        for (int idx = 0; idx < 10; ++idx) {
            const int j = (idx + 1) >> 1;  // idx odd: aligned word j; idx even: odd pair (word j, word j + 1)
            const uint32_t dv = (idx & 1) ? d[j] : odd_pair(d[j], d[j + 1]);
            const uint32_t lv = (idx & 1) ? l[j] : odd_pair(l[j], l[j + 1]);
            m[idx] = pmin(dv, 0xffffffffu - pmin(lv ^ C, SPLAT16(1)) * 0xfffeu);
        }
        uint32_t ta[5], tb[5];  // 5-window maxima of this row as tap-1 row (R1 row k) and as tap-2 row (R1 row k - 3)
        if (!kBorder) {
            uint32_t W[6];  // W_s = max(m[s .. s+4]): tap-1 windows are W_0..W_4, tap-2 windows W_1..W_5
#pragma unroll
            for (int s = 0; s < 6; ++s) W[s] = pmax3(pmax3(m[s], m[s + 1], m[s + 2]), m[s + 3], m[s + 4]);
#pragma unroll
            for (int b = 0; b < 5; ++b) { ta[b] = W[b]; tb[b] = W[b + 1]; }
        } else {
            // R1 columns outside the image are excluded: each tap is masked with the in-image lanes of ITS R1 column
            uint32_t t1[9], t2[9];
#pragma unroll
            for (int jj = 0; jj < 9; ++jj) { t1[jj] = m[jj] & cm[jj]; t2[jj] = m[jj + 1] & cm[jj]; }
#pragma unroll
            for (int b = 0; b < 5; ++b) {
                ta[b] = pmax3(pmax3(t1[b], t1[b + 1], t1[b + 2]), t1[b + 3], t1[b + 4]);
                tb[b] = pmax3(pmax3(t2[b], t2[b + 1], t2[b + 2]), t2[b + 3], t2[b + 4]);
            }
        }
        if (k >= 3) {  // R1 row i = k - 3 (image row gy - 4 + i): tap-1 row k - 3 (waiting in ha), tap-2 row k
            const int i = k - 3;
            const int gr = gy - 4 + i;
            const bool rin = gr >= 0 && gr < rows;  // R1 rows outside the image are excluded
#pragma unroll
            for (int b = 0; b < 5; ++b) ring[i % 5][b] = rin ? pmax(ha[k % 3][b], tb[b]) : 0u;
        }
        if (k <= 8) {
#pragma unroll
            for (int b = 0; b < 5; ++b) ha[k % 3][b] = ta[b];
        }
        if (k >= 7) {
            // H rows i = k-7 .. k-3 are complete: R2 of q row qi = k - 7 (image row gy - 2 + qi), then the erosion over b
            const int qi = k - 7;
            const int gq = gy - 2 + qi;
            if (gq >= 0 && gq < rows) {
                uint32_t e = 0xffffffffu;
#pragma unroll
                for (int b = 0; b < 5; ++b) {
                    uint32_t r2 = pmax3(pmax3(ring[0][b], ring[1][b], ring[2][b]), ring[3][b], ring[4][b]);
                    if (kBorder) r2 |= ~lanes_inside(gx - 2 + b, cols);  // q columns outside the image do not take part in the min
                    e = pmin(e, r2);
                }
                out = pmin(out, e);
            }
        }
    }
    return out;
}

// ---- per-superpixel formulation of the guided stage: one warp per label, lanes = word columns, rows slide through
// registers, horizontal neighbours come from warp shuffles.  For a label c the masked image, its 2-tap dilation, the
// separable 5x5 dilation and erosion are computed over the bounding box of c inside the tile (plus the footprint halo),
// i.e. ~(22+11) x (11+5) words instead of 120 masked words for every one of its ~160 output words.
constexpr int kLabSlots = 512;  // hash table slots for the labels of a tile; more than 3/4 full: the tile falls back to guided_word
struct LabelTable {
    unsigned key[kLabSlots];
    int r0[kLabSlots], r1[kLabSlots], w0[kLabSlots], w1[kLabSlots];
    int list[kLabSlots];
    int n, overflow;
};

__device__ __forceinline__ int label_slot(LabelTable* T, unsigned lab) {
    unsigned h = (lab * 40503u) & (kLabSlots - 1);
    for (int probe = 0; probe < kLabSlots; ++probe) {
        const unsigned old = atomicCAS(&T->key[h], 0xffffffffu, lab);
        if (old == 0xffffffffu || old == lab) return (int)h;
        h = (h + 1) & (kLabSlots - 1);
    }
    T->overflow = 1;
    return -1;
}

__device__ __forceinline__ void label_run(LabelTable* T, unsigned lab, int r, int wa, int wb) {
    const int s = label_slot(T, lab);
    if (s < 0) return;
    atomicMin(&T->r0[s], r);
    atomicMax(&T->r1[s], r);
    atomicMin(&T->w0[s], wa);
    atomicMax(&T->w1[s], wb);
}

// 5-window of a word given its left and right neighbour words (both packed lanes)
template <bool kIsMax>
__device__ __forceinline__ uint32_t h5_word(uint32_t l, uint32_t c, uint32_t r) {
    return pext3<kIsMax>(pext3<kIsMax>(l, odd_pair(l, c), c), odd_pair(c, r), r);
}

// All output pixels of label c inside its bounding box [r0, r1] x [w0, w1] (region rows / words), by kW lanes: a whole warp
// (kW = 32: chunks of 27 output words), or half a warp (kW = 16, boxes up to 11 words wide: two superpixels per warp, the
// shuffles stay inside the half).  Lanes of a half without work (c == 0xffffffff) just keep step.
template <int kW>
__device__ __forceinline__ void guided_label_warp(const uint32_t* __restrict__ A, const uint32_t* __restrict__ LB, uint32_t* __restrict__ B,
                                                  int pitchw, unsigned c, int r0, int r1, int w0, int w1, int n_rows_max, int gy0, int gx0,
                                                  int rows, int cols) {
    const int lane = threadIdx.x & (kW - 1);
    constexpr int kOut = kW - 5;  // output words per chunk: 2 footprint words on the left, 3 on the right
    const uint32_t C2 = c * 0x00010001u;
    const bool idle = c == 0xffffffffu;
    uint16_t* Bh = reinterpret_cast<uint16_t*>(B);
    const int n_chunks = kW == 32 ? (w1 - w0 + kOut) / kOut : 1;  // both halves of a paired warp run one chunk
    for (int ch = 0; ch < n_chunks; ++ch) {
        const int wc = w0 + ch * kOut;
        const int nout = min(kOut, w1 - wc + 1);
        const int w = wc - 2 + lane;
        const bool active = !idle && lane < nout + 5;
        const bool writer = !idle && lane >= 2 && lane < 2 + nout;
        const uint32_t colmask = active ? lanes_inside(gx0 + 2 * w, cols) : 0u;
        uint32_t t1a = 0u, t1b = 0u, t1c = 0u;                    // tap-1 words of the last three masked rows (newest first)
        uint32_t ra = 0u, rb = 0u, rc = 0u, rd = 0u;              // last four R1 rows (newest first)
        uint32_t ea = 0xffffffffu, eb = 0xffffffffu, ec = 0xffffffffu, ed = 0xffffffffu;  // last four eroded rows
        for (int j = 0; j < n_rows_max + 12; ++j) {  // masked row k = r0 - 5 + j (the longer box of a pair sets the trip count)
            const int k = r0 - 5 + j;
            const bool in_box = k <= r1 + 6;
            uint32_t m = 0u;
            if (active && in_box) {
                const uint32_t dv = A[k * pitchw + w], lv = LB[k * pitchw + w];
                m = pmin(dv, 0xffffffffu - pmin(lv ^ C2, SPLAT16(1)) * 0xfffeu);  // same label: the pixel; other: hole; outside: absent
            }
            const uint32_t ms = __shfl_down_sync(0xffffffffu, m, 1, kW);
            // R1 row i = k - 2: tap 1 = pixels (x+1, x+2) of masked row i - 1 = k - 3, tap 2 = pixels (x+2, x+3) of masked row k
            const int gi = gy0 + k - 2;
            const uint32_t r1w = (gi >= 0 && gi < rows) ? (pmax(t1c, ms) & colmask) : 0u;  // R1 outside the image is excluded
            t1c = t1b; t1b = t1a; t1a = odd_pair(m, ms);
            // vertical dilation: R1 rows i-4 .. i  ->  row i - 2 = k - 4
            const uint32_t vd = pmax3(pmax3(rd, rc, rb), ra, r1w);
            rd = rc; rc = rb; rb = ra; ra = r1w;
            // horizontal dilation -> R2 at q row k - 4; q outside the image does not take part in the erosion
            uint32_t h = h5_word<true>(__shfl_up_sync(0xffffffffu, vd, 1, kW), vd, __shfl_down_sync(0xffffffffu, vd, 1, kW));
            const int gq = gy0 + k - 4;
            h = (gq >= 0 && gq < rows) ? (h | ~colmask) : 0xffffffffu;
            // horizontal erosion, then vertical erosion over q rows k-8 .. k-4  ->  output row k - 6
            const uint32_t e = h5_word<false>(__shfl_up_sync(0xffffffffu, h, 1, kW), h, __shfl_down_sync(0xffffffffu, h, 1, kW));
            const uint32_t o = pmin3(pmin3(ed, ec, eb), ea, e);
            ed = ec; ec = eb; eb = ea; ea = e;
            const int orow = k - 6;
            if (writer && in_box && orow >= r0) {
                const uint32_t lw = LB[orow * pitchw + w];
                if ((lw & 0xffffu) == c) Bh[(orow * pitchw + w) * 2] = (uint16_t)(o & 0xffffu);
                if ((lw >> 16) == c) Bh[(orow * pitchw + w) * 2 + 1] = (uint16_t)(o >> 16);
            }
        }
    }
}

// kPerLabel: one warp per superpixel, GTL threads, DCMT_GUIDED_CTAS CTAs per SM (two of 512 on 71-row tiles beat one of 1024 on
// 88 rows by 10 %: the barriers of one CTA are covered by the other); tiles whose labels overflow the table set their flag and
// leave.  !kPerLabel: every word on its own (guided_word), 256 threads, two CTAs per SM; runs for flagged tiles only
// unless g.per_label == 0 (A/B switch).
template <bool kPerLabel, int GT>
__global__ void __launch_bounds__(GT, kPerLabel ? DCMT_GUIDED_CTAS : 2) k_q8_guided_front(GuidedArgs g) {
    DCMT_DYN_SMEM(uint32_t, smem);
    const FrontArgs& a = g.f;
    const int th = a.th, tw = a.tw, rows = a.rows, cols = a.cols;
    Tile t;
    t.RH = th + FU + FD;
    t.RQ = tw / 8 + FLQ + FRQ;
    t.pitchw = t.RQ * 4;
    const int plane = t.RH * t.pitchw;
    uint32_t* A = smem + 4;       // encoded image; later the vertical half of dilate7
    uint32_t* B = A + plane;      // result of the guided stage (the closed image D)
    uint32_t* LB = B + plane + 4; // labels, two uint16 per word (0xffff = no valid label)
    LabelTable* T = reinterpret_cast<LabelTable*>(LB + plane + 4);
    const int frame = blockIdx.z;
    int* tile_flag = g.tile_flags + ((size_t)frame * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;
    if (!kPerLabel && g.per_label && *tile_flag == 0) return;  // the per-label kernel has done this tile
    const int y0 = blockIdx.y * th, x0 = blockIdx.x * tw;
    const int gy0 = y0 - FU, gx0 = x0 - FLQ * 8;
    t.rlo = max(0, -gy0);
    t.rhi = min(t.RH, rows - gy0);
    tile_columns(t, gx0, cols);
    const ptrdiff_t origin = (ptrdiff_t)frame * (ptrdiff_t)a.in_fstride + ((ptrdiff_t)gy0 * (ptrdiff_t)a.in_pitch + gx0);

    float bad = 0.0f;
    if (a.in16 && a.codes) front_load<true, false, true>(a, a.in16 + origin, A, B, t, gx0, bad);
    else if (a.in16) front_load<true, false>(a, a.in16 + origin, A, B, t, gx0, bad);
    else if (a.validate) front_load<false, true>(a, a.in + origin, A, B, t, gx0, bad);
    else front_load<false, false>(a, a.in + origin, A, B, t, gx0, bad);
    // labels of the region (cells outside the image are never looked at: their image value is absent)
    {
        const int32_t* lab = g.labels + (size_t)frame * rows * cols;
        const int nk = g.n_clusters;
        const bool lab_vec2 = (cols & 1) == 0 && (reinterpret_cast<uintptr_t>(g.labels) & 7) == 0;  // every word of every frame 8-byte aligned
        for (int i = threadIdx.x; i < t.RH * t.pitchw; i += GT) {
            const int r = fast_div(i, a.i_half.magic);  // i_half.nq == pitchw here (see q8_run_guided_front)
            const int w = i - r * t.pitchw;
            const int gy = gy0 + r, gx = gx0 + 2 * w;
            uint32_t lo = 0xffffu, hi = 0xffffu;
            if (gy >= 0 && gy < rows) {
                if (lab_vec2 && gx >= 0 && gx + 1 < cols) {  // both pixels of the word in one 8-byte load (gx is even)
                    const int2 v = __ldg(reinterpret_cast<const int2*>(lab + (size_t)gy * cols + gx));
                    if (v.x >= 0 && v.x < nk) lo = (uint32_t)v.x;
                    if (v.y >= 0 && v.y < nk) hi = (uint32_t)v.y;
                } else {
                    if (gx >= 0 && gx < cols) { const int v = __ldg(lab + (size_t)gy * cols + gx); if (v >= 0 && v < nk) lo = (uint32_t)v; }
                    if (gx + 1 >= 0 && gx + 1 < cols) { const int v = __ldg(lab + (size_t)gy * cols + gx + 1); if (v >= 0 && v < nk) hi = (uint32_t)v; }
                }
            }
            LB[i] = lo | (hi << 16);
        }
    }
    if (kPerLabel) {
        for (int i = threadIdx.x; i < kLabSlots; i += GT) {
            T->key[i] = 0xffffffffu;
            T->r0[i] = 0x7fffffff; T->r1[i] = -1; T->w0[i] = 0x7fffffff; T->w1[i] = -1;
        }
        if (threadIdx.x == 0) { T->n = 0; T->overflow = 0; }
    }
    if (__syncthreads_or(bad != 0.0f)) {  // not strict q8: this frame is redone by the generic pipeline
        if (threadIdx.x == 0) a.ctr[frame].needs_generic = 1;
        return;
    }
    if (kPerLabel) {
        // ---- which superpixels have pixels in the needed area (rows core +- 3, words 2 .. (tw + 10) / 2), and where: every thread
        //      walks 8 words of a row and reports runs of one label (a few atomics per run, not per pixel)
        const int w_lo = 2, nw = tw / 2 + 4, nch = (nw + 7) / 8;
        const int rb = max(FU - 3, t.rlo), re = min(FU + th + 3, t.rhi);
        for (int it = threadIdx.x; it < (re - rb) * nch; it += GT) {
            const int rr = it / nch, ch = it - rr * nch;
            const int r = rb + rr, wa = w_lo + 8 * ch, wb = min(wa + 8, w_lo + nw);
            unsigned cur = 0xffffu;
            int run0 = 0;
            for (int w = wa; w < wb; ++w) {
                const uint32_t C = LB[r * t.pitchw + w];
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                    const unsigned lab = half ? (C >> 16) : (C & 0xffffu);  // 0xffff: no label or outside the image
                    if (lab != cur) {
                        if (cur != 0xffffu) label_run(T, cur, r, run0, half ? w : w - 1);
                        cur = lab;
                        run0 = w;
                    }
                }
            }
            if (cur != 0xffffu) label_run(T, cur, r, run0, wb - 1);
        }
        __syncthreads();
        for (int i = threadIdx.x; i < kLabSlots; i += GT)
            if (T->key[i] != 0xffffffffu) T->list[atomicAdd(&T->n, 1)] = i;
        // pixels without a label keep their own value; the labelled lanes are written by the label warps below
        for (int it = threadIdx.x; it < (re - rb) * nw; it += GT) {
            const int rr = fast_div(it, a.m_core.magic);
            const int w = w_lo + (it - rr * nw), r = rb + rr;
            const uint32_t C = LB[r * t.pitchw + w];
            const uint32_t keep = (((C & 0xffffu) == 0xffffu) ? 0x0000ffffu : 0u) | (((C >> 16) == 0xffffu) ? 0xffff0000u : 0u);
            B[r * t.pitchw + w] = A[r * t.pitchw + w] & keep & lanes_inside(gx0 + 2 * w, cols);
        }
        __syncthreads();
        if (T->overflow || T->n > kLabSlots * 3 / 4) {  // too many distinct labels for the table: the word-by-word kernel takes the tile
            if (threadIdx.x == 0) *tile_flag = 1;
            return;
        }
        // two superpixels per warp where both boxes fit half a warp (11 words: the usual case at step 18), else one
        const int warp = threadIdx.x >> 5, half = (threadIdx.x >> 4) & 1;
        for (int e = 2 * warp; e < T->n; e += 2 * (GT / 32)) {
            const int sa = T->list[e], sb = e + 1 < T->n ? T->list[e + 1] : -1;
            const int ha = T->r1[sa] - T->r0[sa] + 1, hb = sb >= 0 ? T->r1[sb] - T->r0[sb] + 1 : 0;
            const bool narrow = T->w1[sa] - T->w0[sa] < 11 && (sb < 0 || T->w1[sb] - T->w0[sb] < 11);
            if (narrow) {
                const int s_ = half ? sb : sa;
                if (s_ >= 0) guided_label_warp<16>(A, LB, B, t.pitchw, T->key[s_], T->r0[s_], T->r1[s_], T->w0[s_], T->w1[s_], max(ha, hb), gy0, gx0, rows, cols);
                else guided_label_warp<16>(A, LB, B, t.pitchw, 0xffffffffu, 5, 5, 2, 2, max(ha, hb), gy0, gx0, rows, cols);
            } else {
                guided_label_warp<32>(A, LB, B, t.pitchw, T->key[sa], T->r0[sa], T->r1[sa], T->w0[sa], T->w1[sa], ha, gy0, gx0, rows, cols);
                if (sb >= 0) guided_label_warp<32>(A, LB, B, t.pitchw, T->key[sb], T->r0[sb], T->r1[sb], T->w0[sb], T->w1[sb], hb, gy0, gx0, rows, cols);
            }
        }
    }
    // ---- the guided stage on rows core +- 3, pixels core -4 .. +3 (what dilate7 reads); words 2 .. (tw + 10) / 2.
    //      (Handling words whose two pixels share a label on a cheaper path, with the others compacted into a list, was
    //      measured: +6 % with real SLIC labels, nothing with jittered ones, and it costs the second CTA per SM.)
    if (!kPerLabel) {
        const int w_lo = 2, nw = tw / 2 + 4;
        const int rb = max(FU - 3, t.rlo), re = min(FU + th + 3, t.rhi);
        // every R1 / q column any item of this tile touches lies inside the image?
        const bool cols_inside = gx0 + 2 * w_lo - 4 >= 0 && gx0 + 2 * (w_lo + nw - 1) + 1 + 5 < cols;
        const int n_items = (re - rb) * nw;
        for (int it = threadIdx.x; it < n_items; it += GT) {
            const int rr = fast_div(it, a.m_core.magic);  // m_core.nq == nw here
            const int w = w_lo + (it - rr * nw), r = rb + rr;
            const int gy = gy0 + r, gx = gx0 + 2 * w;
            const uint32_t inside = lanes_inside(gx, cols);
            uint32_t res = 0u;
            if (inside) {
                const uint32_t C = LB[r * t.pitchw + w], dw = A[r * t.pitchw + w];
                // lanes without a valid label keep their own value (:82 only visits pixels of some superpixel)
                const uint32_t keep = (((C & 0xffffu) == 0xffffu) ? 0x0000ffffu : 0u) | (((C >> 16) == 0xffffu) ? 0xffff0000u : 0u);
                res = dw;
                if (keep != 0xffffffffu) {
                    const uint32_t gw = cols_inside ? guided_word<false>(A, LB, t.pitchw, r, w, C, gy, gx, rows, cols)
                                                    : guided_word<true>(A, LB, t.pitchw, r, w, C, gy, gx, rows, cols);
                    res = (dw & keep) | (gw & ~keep);
                }
                res &= inside;
            }
            B[r * t.pitchw + w] = res;
        }
    }
    __syncthreads();
    // ---- vertical half of dilate7 (:88-90 of img_completion.cpp, :106-108 here) on the core rows: B -> A
    {
        const int rb = max(FU, t.rlo), re = min(FU + th, t.rhi);
        const int nw = tw / 2 + 4, n_items = (re - rb) * nw;
        for (int it = threadIdx.x; it < n_items; it += GT) {
            const int rr = fast_div(it, a.m_core.magic);
            const int off = (rb + rr) * t.pitchw + 2 + (it - rr * nw);
            const uint32_t* p = B + off;
            const int pw = t.pitchw;
            A[off] = pmax3(pmax3(p[-3 * pw], p[-2 * pw], p[-pw]), pmax3(p[0], p[pw], p[2 * pw]), p[3 * pw]);
        }
    }
    __syncthreads();
    // ---- horizontal half of dilate7, hole fill, store the core, column keys: as in k_q8_front
    uint16_t* mid = a.mid + (size_t)frame * a.mid_fstride;
    {
        const int cq = tw / 8;
        const int rend = min(th, rows - y0);
        for (int it = threadIdx.x; it < rend * cq; it += GT) {
            const int r = fast_div(it, a.m_pass.magic);  // m_pass.nq == cq here
            const int q = it - r * cq;
            const int gx = x0 + q * 8;
            if (gx >= cols) continue;
            const int off = ((r + FU) * t.RQ + q + FLQ) * 4;
            const uint4 tt = h7_max_quad(A + off);
            uint4 d = lds4(B + off);
            d.x = fill_holes(d.x, tt.x);
            d.y = fill_holes(d.y, tt.y);
            d.z = fill_holes(d.z, tt.z);
            d.w = fill_holes(d.w, tt.w);
            sts4(B + off, d);
            *reinterpret_cast<uint4*>(mid + (size_t)(y0 + r) * a.mid_pitch + gx) = d;
        }
    }
    __syncthreads();
    const uint16_t* Bh = reinterpret_cast<const uint16_t*>(B);
    const int hrows = min(th, rows - y0);
    for (int c2 = threadIdx.x; c2 < 2 * tw; c2 += GT) {
        const int col = c2 >> 1, from_bottom = c2 & 1;
        const int gx = x0 + col;
        if (gx >= cols) continue;
        const uint16_t* p = Bh + (size_t)FU * t.pitchw * 2 + FLQ * 8 + col;
        if (!from_bottom) {
            for (int cy = 0; cy < hrows; ++cy) {
                const uint32_t e = p[(size_t)cy * t.pitchw * 2];
                if (e >= E_VALID_MIN) {
                    atomicMin(a.col_first + (size_t)frame * a.mid_pitch + gx, ((uint32_t)(y0 + cy) << 16) | e);
                    break;
                }
            }
        } else {
            for (int cy = hrows - 1; cy >= 0; --cy) {
                const uint32_t e = p[(size_t)cy * t.pitchw * 2];
                if (e >= E_VALID_MIN) {
                    atomicMax(a.col_last + (size_t)frame * a.mid_pitch + gx, ((uint32_t)(y0 + cy) << 16) | e);
                    break;
                }
            }
        }
    }
}

// set-up of a front launch in one kernel: the per-column keys and -- unless the caller did it (ctr == nullptr) -- the per-frame counters
// (n >= n_frames: a frame has at least one column)
__global__ void k_q8_init_cols(uint32_t* first, uint32_t* last, size_t n, FrameCounters* ctr, int n_frames) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { first[i] = 0xffffffffu; last[i] = 0u; }
    if (ctr && i < (size_t)n_frames) { ctr[i] = FrameCounters{}; ctr[i].path = 1; }
}

// debugging / test aid: decode a uint16 plane back to float metres in inverted space
__global__ void k_q8_decode(const uint16_t* __restrict__ mid, size_t mid_pitch, float* __restrict__ out, int rows, int cols) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= cols || y >= rows) return;
    const uint32_t e = mid[(size_t)y * mid_pitch + x];
    out[(size_t)y * cols + x] = e == 0 ? -FLT_MAX : (float)(e - 1) * (1.0f / 256.0f);
}

// ------------------------------------------------------------------------------------------------
// k_q8_tail.  Region = core + 19 rows up/down and 24 columns (3 quads) left/right: 15 (one effective 31x31
// fill) + 2 (median) + 2 (Gaussian) = 19.  Two shared-memory planes: A = image, B = vertical 16-row maxima,
// later the median image.
// ------------------------------------------------------------------------------------------------
constexpr int TV = 19, TQ = 3;   // rows up/down, quads left/right
constexpr int kRemCap = 256;     // words still holding a hole after the first fill that are resolved from the list (more: all scan words are visited)
constexpr int kListCap = 3072;   // hole quads kept for the lazy horizontal fill; more than that: all words are processed

struct TailArgs {
    const uint16_t* mid;
    size_t mid_pitch, mid_fstride;
    const uint32_t* col_first;
    const uint32_t* col_last;
    FrameCounters* ctr;
    void* out;                      // float32, or KITTI uint16 for k_q8_tail<false, true>
    size_t out_pitch, out_fstride;  // elements of the output type
    int rows, cols, th, tw, blur, vec_ok;
    int one;          // the constant 1, opaque to the compiler (see other_of_pair)
    int use_tma;      // tile load by one TMA box copy (else 16-byte cp.async per thread)
    ItemsDesc i_load, i_vert, i_scan, i_scanw, i_med, i_gauss;  // row lengths RQ, pitchw, SQ, 4 SQ, MI, NP
    ItemsDesc i_vert2; // row length pitchw / 2: pairs of word columns (vertical maxima)
    ItemsDesc i_medr;  // row length tw / 2 + 2: one item = one word column x med_len rows (shared-work median)
    int med_len, med_segs;
    uint32_t e_hundred;  // code of the constant 100.0: E_HUNDRED (strict q8), kRankHundred (dictionary codes)
    const float* lut;    // dictionary of the frames (kRank): lut[slot * kRankMaxValid + code - kRankFirstCode]
    long long* prof;  // optional: 16 clock64() stamps per CTA (debugging aid)
};

// The element of {a, b} that is not lo = min(a, b), for both packed lanes at once: a + b - lo as ONE 32-bit
// expression is exact (the lane results fit 16 bits, so the carries between the lanes cancel).  Min/max of every
// flavour runs on the ALU pipe at 64 lanes/clk/SM (tools/pipe_bench.cu); integer multiply-add runs on the FMA
// pipe in parallel, so a compare-exchange written this way costs one ALU-pipe slot instead of two.  The multiplier
// is an opaque 1 so that the additions are emitted as IMAD (FMA pipe) and not folded into an ALU-pipe IADD3.
__device__ __forceinline__ uint32_t other_of_pair(uint32_t a, uint32_t b, uint32_t lo, uint32_t one) {
    return a * one + (b * one - lo);
}

#ifndef DCMT_OTH_NUM
#define DCMT_OTH_NUM 0  // of every DCMT_OTH_DEN compare-exchanges of the merge networks, this many take their maximum on the ALU pipe
#endif
#ifndef DCMT_OTH_DEN
#define DCMT_OTH_DEN 1
#endif
struct PackedOps {
    uint32_t one;
    __device__ __forceinline__ uint32_t other(uint32_t a, uint32_t b, uint32_t lo) const { return other_of_pair(a, b, lo, one); }
    template <int I>
    __device__ __forceinline__ uint32_t oth(uint32_t a, uint32_t b, uint32_t lo) const {
        return (I % DCMT_OTH_DEN) < DCMT_OTH_NUM ? pmax(a, b) : other_of_pair(a, b, lo, one);
    }
    static __device__ __forceinline__ uint32_t mn(uint32_t a, uint32_t b) { return pmin(a, b); }
    static __device__ __forceinline__ uint32_t mx(uint32_t a, uint32_t b) { return pmax(a, b); }
    static __device__ __forceinline__ uint32_t mn3(uint32_t a, uint32_t b, uint32_t c) { return pmin3(a, b, c); }
    static __device__ __forceinline__ uint32_t mx3(uint32_t a, uint32_t b, uint32_t c) { return pmax3(a, b, c); }
};

template <bool kOnFma>
__device__ __forceinline__ void pcswap(uint32_t& a, uint32_t& b, uint32_t one) {
    const uint32_t lo = pmin(a, b);
    b = kOnFma ? other_of_pair(a, b, lo, one) : pmax(a, b);
    a = lo;
}
// optimal 9-comparator sort of five packed words (both lanes independently).  Five of the nine maxima are computed
// on the FMA pipe, four on the ALU pipe: with the selection network's own mix this loads both pipes equally.
__device__ __forceinline__ void sort5(uint32_t (&v)[5], uint32_t one) {
    pcswap<true>(v[0], v[1], one); pcswap<false>(v[3], v[4], one); pcswap<true>(v[2], v[4], one);
    pcswap<false>(v[2], v[3], one); pcswap<true>(v[0], v[3], one); pcswap<false>(v[0], v[2], one);
    pcswap<true>(v[1], v[4], one); pcswap<false>(v[1], v[3], one); pcswap<true>(v[1], v[2], one);
}

// lanes equal to 1 (holes) -> 0xffff mask per lane
__device__ __forceinline__ uint32_t hole_mask(uint32_t w) {
    return (((w & 0xffffu) == 1u) ? 0x0000ffffu : 0u) | (((w >> 16) == 1u) ? 0xffff0000u : 0u);
}

// q16 output value (already inverted, < 2^23) -> float, exact: (2^23 + o) / 2^16 - 128
__device__ __forceinline__ float finish_px(uint32_t o) {
    return fmaf(__uint_as_float(0x4b000000u + o), 1.0f / 65536.0f, -128.0f);
}

// q16 output value -> KITTI uint16 (metres * 256): o / 256 rounded half to even, i.e. cvRound(finish_px(o) * 256) (< 2^15,
// no saturation needed).  With blur none o = 6553600 - 256 (e - 1), so u = 25600 - (e - 1) and u / 256 == finish_px(o).
__device__ __forceinline__ uint32_t finish_u16(uint32_t o) { return (o + 127u + ((o >> 8) & 1u)) >> 8; }

// 31-wide horizontal max of the vertical maxima for word w of row r (B holds 16-row maxima: rows r-15..r and r..r+15)
__device__ __forceinline__ uint32_t hmax31(const uint32_t* __restrict__ B, int pitchw, int r, int w) {
    const uint32_t* b0 = B + (r - 15) * pitchw + w;
    const uint32_t* b1 = B + r * pitchw + w;
    uint32_t m = 0u;
#pragma unroll
    for (int j = -7; j <= 7; ++j) m = pmax3(m, b0[j], b1[j]);
    // m.lo / m.hi hold the maxima over the even / odd columns of words w-7 .. w+7; both output lanes need both
    // (lane swap), plus column 2w-15 for the low lane only and column 2w+16 for the high lane only
    return pmax3(m, __byte_perm(m, m, 0x1032), odd_pair(pmax(b0[-8], b1[-8]), pmax(b0[8], b1[8])));
}


// ---- A8 median 5x5 (:170), shared-work form (tools/median_rows_scheme.py).  One item = one packed word column x a run
// of rows.  Per image row the five pixels of the window (both lanes: W[w-1], the odd pair, W[w], the odd pair, W[w+1])
// are sorted once: S[y], used by the five outputs whose window holds row y.  Going down the rows two at a time,
//     PP[q]    = merge(S[q], S[q+1])                         used by four outputs
//     QQ[q]    = ranks 7..12 of merge(PP[q], PP[q+2])        the only elements of rows q..q+3 that can be the median
//     out[q+1] = rank 5 of (QQ[q], S[q-1]),   out[q+2] = rank 5 of (QQ[q], S[q+4])
// i.e. 9 + 13/2 + 24/2 comparators + 8 min/max per output word instead of 13.5 + 54.  The sorted rows and pair merges
// rotate through registers with periods 3 and 2, so six steps are written out and nothing is ever moved.
struct MedianRun {
    uint32_t P[2][10];  // PP[q], PP[q+2] alternate
    uint32_t O[3][5];   // S of the odd rows q-1, q+1, q+3
    uint32_t E[5];      // S[q+2], later S[q+4]
};
__device__ __forceinline__ void sort_row5(const uint32_t* __restrict__ p, uint32_t (&s)[5], uint32_t one) {
    const uint32_t c0 = p[0], c2 = p[1], c4 = p[2];
    s[0] = c0; s[1] = odd_pair(c0, c2); s[2] = c2; s[3] = odd_pair(c2, c4); s[4] = c4;
    sort5(s, one);
}
// K = step number mod 6.  p points at word w-1 of row q+3; o at word w of row q+1.
template <int K>
__device__ __forceinline__ void median_step(MedianRun& m, const PackedOps& ops, const uint32_t* __restrict__ p, uint32_t* __restrict__ o, int pitchw,
                                            bool two) {
    constexpr int pa = K & 1, pb = pa ^ 1, om = K % 3, on = (K + 2) % 3;
    uint32_t qq[6];
    // S[q-1] (slot om) is needed until the first output is out; S[q+3] goes to slot on != om
    sort_row5(p, m.O[on], ops.one);
    merge_5_5(ops, m.E, m.O[on], m.P[pb]);
    merge_10_10_ranks_7_12(ops, m.P[pa], m.P[pb], qq);
    o[0] = rank5_of_6_5(ops, qq, m.O[om]);
    sort_row5(p + pitchw, m.E, ops.one);
    if (two) o[pitchw] = rank5_of_6_5(ops, qq, m.E);
}

// kU16 (strict q8 only): a.out receives KITTI uint16 instead of float32
template <bool kRank, bool kU16 = false>
__global__ void __launch_bounds__(QTT, DCMT_TAIL_CTAS) k_q8_tail(TailArgs a, const __grid_constant__ TensorMap3D tmap) {
    static_assert(!(kRank && kU16), "uint16 output is served on strict-q8 frames only");
    DCMT_DYN_SMEM(uint32_t, smem);
    const int th = a.th, tw = a.tw, rows = a.rows, cols = a.cols;
    const int RH = th + 2 * TV, RQ = tw / 8 + 2 * TQ, pitchw = RQ * 4;
    uint32_t* A = smem;
    uint32_t* B = smem + RH * pitchw;
    uint16_t* list = reinterpret_cast<uint16_t*>(B + RH * pitchw);
    uint16_t* Ah = reinterpret_cast<uint16_t*>(A);
    uint16_t* Bh = reinterpret_cast<uint16_t*>(B);
    __shared__ int s_count, s_remaining, s_holes_core, s_left_core;
    __shared__ uint16_t s_rem_list[kRemCap];  // words of the scan region that still hold a hole after the first fill
    __shared__ __align__(8) uint64_t s_bar;  // mbarrier the TMA tile load signals
    const int slot = blockIdx.z;
    if (a.ctr[slot].needs_generic) return;  // not strict q8: the generic pipeline redoes this frame
    const int y0 = blockIdx.y * th, x0 = blockIdx.x * tw;
    const int gy0 = y0 - TV, gx0 = x0 - TQ * 8;
    const uint16_t* mid = a.mid + (size_t)slot * a.mid_fstride;
    const bool border = gy0 < 0 || gy0 + RH > rows || gx0 < 0 || gx0 + RQ * 8 > cols;
    if (threadIdx.x == 0) { s_count = 0; s_remaining = 0; s_holes_core = 0; s_left_core = 0; }

    DCMT_STAMP(a, 0);
    // ---- load the A4 plane: ONE TMA box copy (200 x 126 uint16 for the KITTI tiles) issued by one thread; the hardware
    //      zero-fills everything outside the image (0 = absent, exactly what the border cells must hold) and signals
    //      an mbarrier.  The per-column keys of the A5 step are fetched while the copy is in flight.  Fallback (no
    //      tensor map): 16-byte cp.async copies by all threads with the border handled in software.
    Tile t;
    t.RH = RH;
    t.RQ = RQ;
    t.pitchw = pitchw;
    t.rlo = max(0, -gy0);
    t.rhi = min(RH, rows - gy0);
    if (a.use_tma) {
        if (threadIdx.x == 0) tma_bar_init(&s_bar);
        __syncthreads();
        if (threadIdx.x == 0) tma_load_3d(A, &tmap, gx0, gy0, slot, &s_bar, (uint32_t)(RH * pitchw * 4));
    } else {
        tile_columns(t, gx0, cols);
        const uint16_t* mp = mid + ((ptrdiff_t)gy0 * (ptrdiff_t)a.mid_pitch + gx0);
        const int mpitch = (int)a.mid_pitch;
        if (!border) {
            for (Items i(a.i_load); i.r < RH; i.next()) DCMT_CP_ASYNC_16(A + i.lin * 4, mp + (i.r * mpitch + i.q * 8));
        } else {
            for (Items i(a.i_load); i.r < RH; i.next()) {
                if (outside(t, i.r, i.q)) sts4(A + i.lin * 4, splat4(kAbsMax));
                else if (i.q == t.qs) sts4(A + i.lin * 4, blend(__ldg(reinterpret_cast<const uint4*>(mp + (i.r * mpitch + i.q * 8))), t.smask, kAbsMax));
                else DCMT_CP_ASYNC_16(A + i.lin * 4, mp + (i.r * mpitch + i.q * 8));
            }
        }
    }
    // A5 (:103-129): two threads per region column, one per zone (rows <= first, rows >= last)
    const int a5_item = threadIdx.x, a5_c = a5_item >> 1, a5_bottom = a5_item & 1;
    const int a5_gx = gx0 + a5_c;
    const bool a5_live = a5_item < 2 * RQ * 8 && a5_gx >= 0 && a5_gx < cols;
    uint32_t a5_kf = 0xffffffffu, a5_kl = 0u;
    if (a5_live) {
        a5_kf = __ldg(a.col_first + (size_t)slot * a.mid_pitch + a5_gx);
        a5_kl = __ldg(a.col_last + (size_t)slot * a.mid_pitch + a5_gx);
    }
    if (a.use_tma) tma_bar_wait(&s_bar, 0);
    else DCMT_CP_ASYNC_WAIT_ALL();
    __syncthreads();
    DCMT_STAMP(a, 1);
    // rows >= last <- value(last), rows <= first <- value(first) (the second write wins); empty column <- 100
    auto a5_apply = [&](int item, uint32_t kf, uint32_t kl) {
        const int c = item >> 1, bottom = item & 1;
        const bool empty = kf == 0xffffffffu;
        const int first = empty ? rows - 1 : (int)(kf >> 16), last = empty ? 0 : (int)(kl >> 16);
        uint16_t* p = Ah + c;
        if (!bottom) {
            const uint16_t nv = empty ? (uint16_t)a.e_hundred : (uint16_t)(kf & 0xffffu);
            const int r1 = min(RH - 1, first - gy0);
            for (int r = max(0, -gy0); r <= r1; ++r) p[(size_t)r * pitchw * 2] = nv;
        } else {
            const uint16_t mv = empty ? (uint16_t)a.e_hundred : (uint16_t)(kl & 0xffffu);
            const int r1 = min(RH - 1, rows - 1 - gy0);
            for (int r = max(max(0, -gy0), max(last, first + 1) - gy0); r <= r1; ++r) p[(size_t)r * pitchw * 2] = mv;
        }
    };
    if (a5_live) a5_apply(a5_item, a5_kf, a5_kl);
    for (int item = a5_item + QTT; item < 2 * RQ * 8; item += QTT) {  // CTAs with fewer threads than 2 x region columns
        const int gx = gx0 + (item >> 1);
        if (gx >= 0 && gx < cols)
            a5_apply(item, __ldg(a.col_first + (size_t)slot * a.mid_pitch + gx), __ldg(a.col_last + (size_t)slot * a.mid_pitch + gx));
    }
    __syncthreads();
    DCMT_STAMP(a, 2);
    // ---- A6 vertical part: B(r) = max of A over rows r .. r+15 (van Herk / Gil-Werman with blocks of 16 rows).
    //      One item = one word column x one block: suffix maxima of the block's 16 rows stay in registers, the
    //      running prefix maximum of the next 15 rows completes every window.  No intermediate planes, one barrier.
    {
        const int NB = (TV + th + 4 + 15) / 16;  // vertical maxima are needed for rows [0, TV + th + 4)
        // one item = TWO adjacent word columns x one block (8-byte accesses): the phase is bound by shared-memory
        // instructions and latency, and 50 x 8 items fit the CTA's threads in one round where 100 x 8 took two
        for (Items i(a.i_vert2); i.r < NB; i.next()) {
            const int r0 = 16 * i.r;
            const uint32_t* p = A + r0 * pitchw + 2 * i.q;
            uint32_t* o = B + r0 * pitchw + 2 * i.q;
            uint2 sfx[16];
            sfx[15] = lds2(p + 15 * pitchw);
#pragma unroll
            for (int k = 14; k >= 0; --k) {
                const uint2 v = lds2(p + k * pitchw);
                sfx[k] = make_uint2(pmax(v.x, sfx[k + 1].x), pmax(v.y, sfx[k + 1].y));
            }
            sts2(o, sfx[0]);
            uint2 m = make_uint2(0u, 0u);
#pragma unroll
            for (int j = 1; j < 16; ++j) {
                if (r0 + 15 + j < RH) {  // rows past the region are absent
                    const uint2 v = lds2(p + (15 + j) * pitchw);
                    m = make_uint2(pmax(m.x, v.x), pmax(m.y, v.y));
                }
                sts2(o + j * pitchw, make_uint2(pmax(sfx[j].x, m.x), pmax(sfx[j].y, m.y)));
            }
        }
    }
    __syncthreads();
    DCMT_STAMP(a, 3);
    // ---- A6 horizontal part on hole words only (:131-144): scan quads for lanes == 1, ballot/popc-compact the
    //      words that hold a hole into a list, then a 31-wide max of the vertical maxima for those words.
    //      Scan region: rows core +- 4, quads covering columns core +- 8 (a superset of the +- 4 the median needs).
    const int SH = th + 8, SQ = tw / 8 + 2;
    const int sr0 = TV - 4, sq0 = TQ - 1;
    {
        const int n = SH * SQ;
        Items i(a.i_scan);
        constexpr int kScanRounds = 6;
        if (n <= kScanRounds * QTT) {
            // all rounds of a warp first (independent loads and ballots), then ONE reservation per warp in the list
            uint32_t qv[kScanRounds];
            unsigned bal[kScanRounds];
            int total = 0;
#pragma unroll
            for (int k = 0; k < kScanRounds; ++k) {
                bool cand = false;
                qv[k] = 0u;
                if (k * QTT + (int)threadIdx.x < n) {
                    const int qidx = (sr0 + i.r) * RQ + sq0 + i.q;
                    const uint4 v = lds4(A + qidx * 4);
                    // some lane <= 1 (a hole, or absent outside the image)?
                    cand = pmin(pmin(pmin(v.x, v.y), pmin(v.z, v.w)), SPLAT16(2)) != SPLAT16(2);
                    qv[k] = (uint32_t)qidx | (cand ? 0x80000000u : 0u);
                }
                bal[k] = __ballot_sync(0xffffffffu, cand);
                total += __popc(bal[k]);
                i.next();
            }
            if (total) {
                int pos = 0;
                if ((threadIdx.x & 31) == 0) pos = atomicAdd(&s_count, total);
                pos = __shfl_sync(0xffffffffu, pos, 0);
                const unsigned below = (1u << (threadIdx.x & 31)) - 1u;
#pragma unroll
                for (int k = 0; k < kScanRounds; ++k) {
                    const int at = pos + __popc(bal[k] & below);
                    if ((qv[k] & 0x80000000u) && at < kListCap) list[at] = (uint16_t)(qv[k] & 0xffffu);
                    pos += __popc(bal[k]);
                }
            }
        } else {
            for (int base = 0; base < n; base += QTT, i.next()) {
                bool cand = false;
                int qidx = 0;
                if (base + (int)threadIdx.x < n) {
                    qidx = (sr0 + i.r) * RQ + sq0 + i.q;
                    const uint4 v = lds4(A + qidx * 4);
                    cand = pmin(pmin(pmin(v.x, v.y), pmin(v.z, v.w)), SPLAT16(2)) != SPLAT16(2);
                }
                const unsigned bal = __ballot_sync(0xffffffffu, cand);
                if (bal == 0u) continue;
                int pos = 0;
                if ((threadIdx.x & 31) == 0) pos = atomicAdd(&s_count, __popc(bal));
                pos = __shfl_sync(0xffffffffu, pos, 0) + __popc(bal & ((1u << (threadIdx.x & 31)) - 1u));
                if (cand && pos < kListCap) list[pos] = (uint16_t)qidx;
            }
        }
    }
    __syncthreads();
    DCMT_STAMP(a, 4);
    int holes_core = 0, left_core = 0;
    const int n_quads = s_count;
    auto fill_word = [&](int widx) {
        const uint32_t d = A[widx], hm = hole_mask(d);
        if (hm == 0u) return;
        const int r = fast_div(widx, a.i_vert.magic), w = widx - r * pitchw;
        const int sr = r - sr0, sw = w - TQ * 4;
        const bool core = sr >= 4 && sr < 4 + th && sw >= 0 && sw < tw / 2;
        if (core) holes_core += __popc(hm) >> 4;
        const uint32_t nd = (hmax31(B, pitchw, r, w) & hm) | (d & ~hm);
        A[widx] = nd;
        const uint32_t still = hole_mask(nd);
        if (still) {
            if (core) left_core += __popc(still) >> 4;
            const int pos = atomicAdd(&s_remaining, 1);
            if (pos < kRemCap) s_rem_list[pos] = (uint16_t)widx;
        }
    };
    if (n_quads <= kListCap) {
        for (int k = threadIdx.x; k < 4 * n_quads; k += QTT) fill_word(list[k >> 2] * 4 + (k & 3));
    } else {  // cannot happen for tiles up to 96 x 160 (2184 scan quads); kept for larger tiles
        for (Items i(a.i_scanw); i.r < SH; i.next()) fill_word((sr0 + i.r) * pitchw + sq0 * 4 + i.q);
    }
    if (holes_core) atomicAdd(&s_holes_core, holes_core);
    if (left_core) atomicAdd(&s_left_core, left_core);
    __syncthreads();
    if (threadIdx.x == 0) {
        if (s_holes_core) atomicAdd(&a.ctr[slot].holes_after_extrapolation, s_holes_core);
        if (s_left_core) atomicAdd(&a.ctr[slot].holes_after_first_fill, s_left_core);
    }
    // ---- A7 (:146-166): the reference repeats the 31x31 fill until no hole is left.  A hole that survives the first
    //      fill has no valid pixel within 15; pass k of the loop gives it the maximum over the (30 k + 1)-square around
    //      it of the image BEFORE the loop (a fill of fills is a fill with the summed radius, and a pixel is filled by
    //      the first pass whose square reaches a valid pixel).  Such holes are rare, so each is resolved directly: one
    //      warp scans growing squares of the A5 image in global memory (intermediate plane + column keys) until it
    //      meets a valid pixel.  Every tile resolves the holes of its own scan region from the same global data, so
    //      neighbouring tiles agree without talking to each other.
    const int n_rem = s_remaining;
    if (n_rem > 0) {
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = QTT / 32;
        int max_pass = 0;
        auto resolve_word = [&](int widx) {
            const uint32_t d = A[widx];
            if (hole_mask(d) == 0u) return;
            const int r = fast_div(widx, a.i_vert.magic), w = widx - r * pitchw;
            uint32_t nd = d;
#pragma unroll 1
            for (int half_lane = 0; half_lane < 2; ++half_lane) {
                if (((d >> (16 * half_lane)) & 0xffffu) != 1u) continue;
                const int gy = gy0 + r, gx = gx0 + 2 * w + half_lane;
                uint32_t m = 0u;
                int k = 1;
                while (m < E_VALID_MIN) {
                    ++k;
                    const int half = 15 * k;
                    const int r_lo = max(gy - half, 0), r_hi = min(gy + half, rows - 1);
                    const int c_lo = max(gx - half, 0), c_hi = min(gx + half, cols - 1);
                    for (int c = c_lo + lane; c <= c_hi; c += 32) {
                        const uint32_t kf = __ldg(a.col_first + (size_t)slot * a.mid_pitch + c), kl = __ldg(a.col_last + (size_t)slot * a.mid_pitch + c);
                        if (kf == 0xffffffffu) { m = max(m, a.e_hundred); continue; }  // empty column: 100 everywhere (:110)
                        const int first = (int)(kf >> 16), last = (int)(kl >> 16);
                        if (r_lo <= first) m = max(m, kf & 0xffffu);   // rows <= first hold value(first)
                        if (r_hi >= last) m = max(m, kl & 0xffffu);    // rows >= last hold value(last)
                        const uint16_t* col = mid + c;
                        for (int rr = max(r_lo, first + 1); rr <= min(r_hi, last - 1); ++rr) m = max(m, (uint32_t)col[(size_t)rr * a.mid_pitch]);
                    }
#pragma unroll
                    for (int sft = 16; sft >= 1; sft >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, sft));
                    if (r_lo == 0 && c_lo == 0 && r_hi == rows - 1 && c_hi == cols - 1) break;  // whole image scanned
                }
                max_pass = max(max_pass, k);
                nd = half_lane ? ((nd & 0x0000ffffu) | (m << 16)) : ((nd & 0xffff0000u) | m);
            }
            if (lane == 0) A[widx] = nd;
        };
        if (n_rem <= kRemCap) {
            for (int e = warp; e < n_rem; e += nwarps) resolve_word(s_rem_list[e]);
        } else {
            for (int e = warp; e < SH * SQ * 4; e += nwarps) {
                const int sr = e / (SQ * 4);
                resolve_word((sr0 + sr) * pitchw + sq0 * 4 + (e - sr * SQ * 4));
            }
        }
        if (lane == 0 && max_pass > 1) atomicMax(&a.ctr[slot].extra_passes, max_pass - 1);
        __syncthreads();
    }
    DCMT_STAMP(a, 5);
    // ---- BORDER_REPLICATE for the median (:170): copy the nearest image pixel into the cells outside the image
    //      (rows / columns core +- 4).  Only the strips that are outside are visited.
    if (border) {
        const int c_lo = TQ * 8 - 4, c_n = tw + 8;
        const int r_in0 = max(sr0, -gy0), r_in1 = min(sr0 + SH, rows - gy0);          // in-image scan rows [r_in0, r_in1)
        const int c_in0 = max(c_lo, -gx0), c_in1 = min(c_lo + c_n, cols - gx0);        // in-image scan columns
        const int n_rows_out = SH - max(0, r_in1 - r_in0), n_cols_out = c_n - max(0, c_in1 - c_in0);
        // (1) columns outside, rows inside   (2) rows outside, all columns.  Both read in-image cells only (row and
        //     column clamped at once), so the two loops need no barrier between them.
        for (int it = threadIdx.x; it < max(0, r_in1 - r_in0) * n_cols_out; it += QTT) {
            const int rr = it / n_cols_out, k = it - rr * n_cols_out;
            const int r = r_in0 + rr;
            const int c = k < c_in0 - c_lo ? c_lo + k : c_in1 + (k - (c_in0 - c_lo));
            const int cc = clampi(c, c_in0, c_in1 - 1);
            Ah[(size_t)r * pitchw * 2 + c] = Ah[(size_t)r * pitchw * 2 + cc];
        }
        for (int it = threadIdx.x; it < n_rows_out * c_n; it += QTT) {
            const int k = it / c_n, c = c_lo + (it - k * c_n);
            const int r = k < r_in0 - sr0 ? sr0 + k : r_in1 + (k - (r_in0 - sr0));
            const int cr = clampi(r, r_in0, r_in1 - 1);
            if (cr >= 0 && cr < RH) Ah[(size_t)r * pitchw * 2 + c] = Ah[(size_t)cr * pitchw * 2 + clampi(c, c_in0, c_in1 - 1)];
        }
        __syncthreads();
    }
    DCMT_STAMP(a, 6);
#if DCMT_MEDIAN_ROWS
    // ---- A8 median 5x5 (:170): shared-work form, see median_step
    {
        const int MH = th + 4;  // rows core +- 2, words core +- 1 (a.i_medr)
        const int mr0 = TV - 2, mw0 = TQ * 4 - 1;
        const PackedOps ops{(uint32_t)a.one};
        for (Items i(a.i_medr); i.r < a.med_segs; i.next()) {
            int r = mr0 + i.r * a.med_len;  // first output row of the run
            const int rend = min(r + a.med_len, mr0 + MH);
            const uint32_t* p = A + (r - 2) * pitchw + (mw0 + i.q - 1);
            uint32_t* o = B + r * pitchw + (mw0 + i.q);
            MedianRun m;
            // q = r - 1:  S[q-1] -> O[0], S[q] and S[q+1] -> PP[q] = P[0] (S[q+1] kept in O[1]), S[q+2] -> E
            uint32_t s0[5];
            sort_row5(p, m.O[0], ops.one);
            sort_row5(p + pitchw, s0, ops.one);
            sort_row5(p + 2 * pitchw, m.O[1], ops.one);
            merge_5_5(ops, s0, m.O[1], m.P[0]);
            sort_row5(p + 3 * pitchw, m.E, ops.one);
            p += 4 * pitchw;
#pragma unroll 1
            for (;;) {
#define DCMT_MEDIAN_STEP(K)                                            \
    median_step<K>(m, ops, p, o, pitchw, r + 1 < rend);                \
    r += 2; p += 2 * pitchw; o += 2 * pitchw;                          \
    if (r >= rend) break;
                DCMT_MEDIAN_STEP(0) DCMT_MEDIAN_STEP(1) DCMT_MEDIAN_STEP(2) DCMT_MEDIAN_STEP(3) DCMT_MEDIAN_STEP(4) DCMT_MEDIAN_STEP(5)
#undef DCMT_MEDIAN_STEP
            }
        }
    }
#else
    // ---- A8 median 5x5 (:170): one item = four output words of one row.  The six word columns it touches are sorted
    //      once (9 compare-exchanges each, both lanes at once), the odd-aligned pixel pairs between them come from
    //      PRMTs of the sorted columns, and each output is the 54-comparator selection network of median_net.cuh on
    //      its five sorted columns.
    {
        const int MH = th + 4;  // rows core +- 2; items of four words cover core +- 1 word (a.i_med)
        const int mr0 = TV - 2, mw0 = TQ * 4 - 1;
        const PackedOps ops{(uint32_t)a.one};
        for (Items i(a.i_med); i.r < MH; i.next()) {
            const int r = mr0 + i.r, w = mw0 + 4 * i.q;  // output words w .. w+3; columns w-1 .. w+4
            uint32_t col[6][5];
            const uint32_t* p = A + (r - 2) * pitchw + (w - 1);  // w - 1 is even: 8-byte aligned
#pragma unroll
            for (int k = 0; k < 5; ++k) {
                const uint2 p0 = *reinterpret_cast<const uint2*>(p + k * pitchw), p1 = *reinterpret_cast<const uint2*>(p + k * pitchw + 2),
                            p2 = *reinterpret_cast<const uint2*>(p + k * pitchw + 4);
                col[0][k] = p0.x; col[1][k] = p0.y; col[2][k] = p1.x; col[3][k] = p1.y; col[4][k] = p2.x; col[5][k] = p2.y;
            }
#pragma unroll
            for (int j = 0; j < 6; ++j) sort5(col[j], ops.one);
            uint32_t res[4];
            uint32_t oddl[5];  // sorted column of the odd-aligned pair left of the current output word
#pragma unroll
            for (int k = 0; k < 5; ++k) oddl[k] = odd_pair(col[0][k], col[1][k]);
#pragma unroll
            for (int o = 0; o < 4; ++o) {
                uint32_t oddr[5];
#pragma unroll
                for (int k = 0; k < 5; ++k) oddr[k] = odd_pair(col[o + 1][k], col[o + 2][k]);
                uint32_t c[25];
#pragma unroll
                for (int k = 0; k < 5; ++k) {
                    c[k] = col[o][k];
                    c[5 + k] = oddl[k];
                    c[10 + k] = col[o + 1][k];
                    c[15 + k] = oddr[k];
                    c[20 + k] = col[o + 2][k];
                }
                res[o] = median25_sorted_columns(ops, c);
#pragma unroll
                for (int k = 0; k < 5; ++k) oddl[k] = oddr[k];
            }
            uint32_t* q = B + r * pitchw + w;  // w is odd: store as 1 + 2 + 1 words
            q[0] = res[0];
            *reinterpret_cast<uint2*>(q + 1) = make_uint2(res[1], res[2]);
            q[3] = res[3];
        }
    }
#endif
    __syncthreads();
    DCMT_STAMP(a, 7);
    // ---- BORDER_REFLECT_101 for the Gaussian (:179): mirror the median image into the 2 cells beyond each edge.
    //      Columns beyond the edge (rows inside) and whole rows beyond the edge; both read in-image cells only (row and
    //      column mirrored at once), so no barrier is needed between the two loops.
    if (border && a.blur == 1) {
        const int c_lo = TQ * 8 - 2, c_n = tw + 4, r_lo = TV - 2, r_n = th + 4;
        const int r_in0 = max(r_lo, -gy0), r_in1 = min(r_lo + r_n, rows - gy0);
        const int c_in0 = max(c_lo, -gx0), c_in1 = min(c_lo + c_n, cols - gx0);
        // at most 2 columns on each side matter: region columns -gx0-2, -gx0-1 and cols-gx0, cols-gx0+1
        for (int it = threadIdx.x; it < max(0, r_in1 - r_in0) * 4; it += QTT) {
            const int r = r_in0 + (it >> 2), k = it & 3;
            const int gx = k < 2 ? k - 2 : cols + (k - 2);
            const int c = gx - gx0, cc = reflect101(gx, cols) - gx0;
            if (c >= c_lo && c < c_lo + c_n && cc >= c_in0 && cc < c_in1) Bh[(size_t)r * pitchw * 2 + c] = Bh[(size_t)r * pitchw * 2 + cc];
        }
        for (int it = threadIdx.x; it < 4 * c_n; it += QTT) {
            const int k = it / c_n, c = c_lo + (it - k * c_n);
            const int gy = k < 2 ? k - 2 : rows + (k - 2);
            const int r = gy - gy0, cr = reflect101(gy, rows) - gy0;
            const int gxc = gx0 + c;
            const int cs = (gxc < 0 || gxc >= cols) ? reflect101(gxc, cols) - gx0 : c;  // source column inside the image
            if (r >= r_lo && r < r_lo + r_n && cr >= r_in0 && cr < r_in1 && cs >= c_in0 && cs < c_in1)
                Bh[(size_t)r * pitchw * 2 + c] = Bh[(size_t)cr * pitchw * 2 + cs];
        }
        __syncthreads();
    }
    DCMT_STAMP(a, 8);
    if (kRank) {
        // ---- A9 + A10 on dictionary codes: decode with the frame's LUT (the inverted float each code stands for; kRankHundred
        //      = 100.0), 5x5 Gaussian in float32 -- the separable symmetric form OpenCV's float path uses, kernel
        //      [.0625 .25 .375 .25 .0625], rows then columns (:176-179) -- masked copy (:181-188: every pixel is valid here),
        //      final inversion (:191-202).  Every pixel is decoded ONCE (a gather from the LUT in global memory) into a float
        //      plane that takes the place of plane A, dead since the median; it holds half the tile's rows at a time.
        float* out = static_cast<float*>(a.out) + (size_t)slot * a.out_fstride;
        const float* lut = a.lut + (size_t)slot * kRankMaxValid;
        const uint32_t eh = a.e_hundred;
        // (cells of the tile that lie outside the image hold 0 / stale codes and only feed outputs that are never stored: the
        // index is clamped so that they read inside the dictionary)
        auto dec = [&](uint32_t e) -> float { return e == eh ? kMaxDepth : __ldg(lut + min(max((int)e - kRankFirstCode, 0), kRankMaxValid - 1)); };
        auto inv_out = [&](float d) -> float { return d >= 0.1f ? __fsub_rn(kMaxDepth, d) : d; };
        float* F = reinterpret_cast<float*>(A);  // (rows of the half + 4) x (tw + 4) floats
        const int FW = tw + 4, NGR = (th + 3) / 4, NP = tw / 4;
        const int gsplit = (NGR + 1) / 2;  // item rows [0, gsplit) first, then [gsplit, NGR)
        for (int half = 0; half < 2; ++half) {
            const int g0 = half ? gsplit : 0, g1 = half ? NGR : gsplit;
            if (g0 >= g1) break;
            const int fr0 = 4 * g0 - 2, fr_n = 4 * (g1 - g0) + 4;  // core rows fr0 .. fr0 + fr_n - 1 (relative to the core)
            if (a.blur == 1) {
                if (half) __syncthreads();  // the first half's readers are done with F
                for (int it = threadIdx.x; it < fr_n * (FW / 2); it += QTT) {
                    const int rr = it / (FW / 2), wq = it - rr * (FW / 2);
                    const uint32_t w = B[(TV + fr0 + rr) * pitchw + TQ * 4 - 1 + wq];  // pixels core column 2 wq - 2, 2 wq - 1
                    *reinterpret_cast<float2*>(F + rr * FW + 2 * wq) = make_float2(dec(w & 0xffffu), dec(w >> 16));
                }
                __syncthreads();
            }
            for (int it = threadIdx.x; it < (g1 - g0) * NP; it += QTT) {
                const int gr = it / NP, ip = it - gr * NP;
                const int cy0 = (g0 + gr) * 4, gx = x0 + ip * 4;
                if (y0 + cy0 >= rows || gx >= cols) continue;
                float* o = out + (size_t)(y0 + cy0) * a.out_pitch + gx;
                float f[4][4];
                if (a.blur == 1) {
                    float h[8][4];
                    const float* fp = F + (cy0 - 2 - fr0) * FW + ip * 4;  // row cy0 - 2, pixel gx - 2
#pragma unroll
                    for (int k = 0; k < 8; ++k) {  // input rows cy0-2 .. cy0+5, pixels gx-2 .. gx+5
                        const float4 xa = *reinterpret_cast<const float4*>(fp + k * FW), xb = *reinterpret_cast<const float4*>(fp + k * FW + 4);
                        const float xs[8] = {xa.x, xa.y, xa.z, xa.w, xb.x, xb.y, xb.z, xb.w};
#pragma unroll
                        for (int c = 0; c < 4; ++c)
                            h[k][c] = __fadd_rn(__fadd_rn(__fmul_rn(xs[c + 2], 0.375f), __fmul_rn(__fadd_rn(xs[c + 1], xs[c + 3]), 0.25f)),
                                                __fmul_rn(__fadd_rn(xs[c], xs[c + 4]), 0.0625f));
                    }
#pragma unroll
                    for (int j = 0; j < 4; ++j)
#pragma unroll
                        for (int c = 0; c < 4; ++c)
                            f[j][c] = inv_out(__fadd_rn(__fadd_rn(__fmul_rn(h[j + 2][c], 0.375f), __fmul_rn(__fadd_rn(h[j + 1][c], h[j + 3][c]), 0.25f)),
                                                        __fmul_rn(__fadd_rn(h[j][c], h[j + 4][c]), 0.0625f)));
                } else {
                    const uint32_t* p = B + (TV + cy0) * pitchw + TQ * 4 + 2 * ip;
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const uint32_t w0 = p[j * pitchw], w1 = p[j * pitchw + 1];
                        f[j][0] = inv_out(dec(w0 & 0xffffu));
                        f[j][1] = inv_out(dec(w0 >> 16));
                        f[j][2] = inv_out(dec(w1 & 0xffffu));
                        f[j][3] = inv_out(dec(w1 >> 16));
                    }
                }
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    if (cy0 + j >= th || y0 + cy0 + j >= rows) break;
                    float* oj = o + (size_t)j * a.out_pitch;
                    if (gx + 4 <= cols && a.vec_ok) {
                        *reinterpret_cast<float4*>(oj) = make_float4(f[j][0], f[j][1], f[j][2], f[j][3]);
                    } else {
#pragma unroll
                        for (int c = 0; c < 4; ++c)
                            if (gx + c < cols) oj[c] = f[j][c];
                    }
                }
            }
        }
    } else {
    // ---- A9 + A10: 5x5 Gaussian [1 4 6 4 1]^2 / 256 in integer q16 (:176-189), final inversion (:191-202), float32
    //      store.  One item = 4 pixels (two words) x 4 rows: the horizontal [1 4 6 4 1] sums of the 8 rows it touches
    //      come straight from the packed words with 16-bit x 8-bit dot products (IDP.2A), the vertical combination
    //      runs on those 32-bit sums in registers.  Every pixel is valid here (a frame with holes left is redone by
    //      k_q8_fixup), so the masked copy (:181-188) always takes the blurred value and the inversion always
    //      applies:  out16 = 6553600 - (g - 256)  with e = q + 1 and weights summing to 256.  kU16: the same value as
    //      KITTI uint16 (finish_u16), 8-byte stores.
    {
        float* out = static_cast<float*>(a.out) + (size_t)slot * a.out_fstride;
        uint16_t* out16 = static_cast<uint16_t*>(a.out) + (size_t)slot * a.out_fstride;
        const int NGR = (th + 3) / 4;  // items: tw / 4 per row of items (a.i_gauss)
        for (Items i(a.i_gauss); i.r < NGR; i.next()) {
            const int cy0 = i.r * 4, gx = x0 + i.q * 4;
            if (y0 + cy0 >= rows || gx >= cols) continue;
            const uint32_t* p = B + (TV + cy0) * pitchw + TQ * 4 + 2 * i.q;  // row cy0, first word of the pair
            const size_t o_off = (size_t)(y0 + cy0) * a.out_pitch + gx;
            uint32_t f[4][4];
            if (a.blur == 1) {
                uint32_t h[8][4];
#pragma unroll
                for (int k = 0; k < 8; ++k) {  // input rows cy0-2 .. cy0+5
                    const uint32_t* q = p + (k - 2) * pitchw;
                    const uint32_t wa = q[-1], wb = q[0], wc = q[1], wd = q[2];
                    h[k][0] = __dp2a_lo(wa, 0x0401u, __dp2a_lo(wb, 0x0406u, __dp2a_lo(wc, 0x0001u, 0u)));
                    h[k][1] = __dp2a_lo(wa, 0x0100u, __dp2a_lo(wb, 0x0604u, __dp2a_lo(wc, 0x0104u, 0u)));
                    h[k][2] = __dp2a_lo(wb, 0x0401u, __dp2a_lo(wc, 0x0406u, __dp2a_lo(wd, 0x0001u, 0u)));
                    h[k][3] = __dp2a_lo(wb, 0x0100u, __dp2a_lo(wc, 0x0604u, __dp2a_lo(wd, 0x0104u, 0u)));
                }
#pragma unroll
                for (int j = 0; j < 4; ++j)
#pragma unroll
                    for (int c = 0; c < 4; ++c)
                        f[j][c] = 6553856u - ((h[j][c] + h[j + 4][c]) + 4u * (h[j + 1][c] + h[j + 3][c]) + 6u * h[j + 2][c]);
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const uint32_t w0 = p[j * pitchw], w1 = p[j * pitchw + 1];
                    f[j][0] = 6553856u - ((w0 & 0xffffu) << 8);  // 6553600 - ((e - 1) << 8)
                    f[j][1] = 6553856u - ((w0 >> 16) << 8);
                    f[j][2] = 6553856u - ((w1 & 0xffffu) << 8);
                    f[j][3] = 6553856u - ((w1 >> 16) << 8);
                }
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if (cy0 + j >= th || y0 + cy0 + j >= rows) break;  // rows past the core belong to the next tile
                if (kU16) {
                    uint16_t* oj = out16 + o_off + (size_t)j * a.out_pitch;
                    if (gx + 4 <= cols && a.vec_ok) {
                        *reinterpret_cast<uint2*>(oj) = make_uint2(finish_u16(f[j][0]) | finish_u16(f[j][1]) << 16,
                                                                   finish_u16(f[j][2]) | finish_u16(f[j][3]) << 16);
                    } else {
#pragma unroll
                        for (int c = 0; c < 4; ++c)
                            if (gx + c < cols) oj[c] = (uint16_t)finish_u16(f[j][c]);
                    }
                } else {
                    float* oj = out + o_off + (size_t)j * a.out_pitch;
                    if (gx + 4 <= cols && a.vec_ok) {
                        *reinterpret_cast<float4*>(oj) = make_float4(finish_px(f[j][0]), finish_px(f[j][1]), finish_px(f[j][2]), finish_px(f[j][3]));
                    } else {
#pragma unroll
                        for (int c = 0; c < 4; ++c)
                            if (gx + c < cols) oj[c] = finish_px(f[j][c]);
                    }
                }
            }
        }
    }
    }
    DCMT_STAMP(a, 9);
}

// main.cpp:79 `convertTo(CV_32F, 1.0 / 256.0)` for frames the fused kernels do not serve (generic pipeline input)
__global__ void k_u16_to_f32(const uint16_t* __restrict__ in, size_t in_pitch, size_t in_fstride, float* __restrict__ out, int rows, int cols) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y, f = blockIdx.z;
    if (x < cols) out[((size_t)f * rows + y) * cols + x] = (float)in[(size_t)f * in_fstride + (size_t)y * in_pitch + x] * (1.0f / 256.0f);
}

// cv::Mat::convertTo(CV_16U, 256.0) of a CV_32FC1 depth map -- what a caller does in front of cv::imwrite of a KITTI depth
// PNG: u = saturate_cast<uint16_t>(cvRound(v * 256)).  The product is exact (a power-of-two scaling), rounding is half to
// even, the result is clamped to [0, 65535] and NaN gives 0.
__device__ __forceinline__ uint32_t depth_u16(float v) {
    const float s = v * 256.0f;
    if (!(s > 0.0f)) return 0u;  // NaN, zeros, negatives
    return s >= 65535.0f ? 65535u : (uint32_t)rintf(s);
}

// pitched, batched float32 -> uint16 by the rule above; a thread converts 4 pixels of a row (one 16-byte load and one
// 8-byte store when `vec`: both layouts aligned), pixel by pixel at the ragged end.  Rows beyond the grid are strided.
__global__ void k_depth_to_u16(const float* __restrict__ in, size_t in_pitch, size_t in_fstride, uint16_t* __restrict__ out,
                               size_t out_pitch, size_t out_fstride, int rows, int cols, int vec) {
    const int x = (blockIdx.x * blockDim.x + threadIdx.x) * 4, f = blockIdx.z;
    if (x >= cols) return;
    for (int y = blockIdx.y; y < rows; y += gridDim.y) {
        const float* i = in + (size_t)f * in_fstride + (size_t)y * in_pitch + x;
        uint16_t* o = out + (size_t)f * out_fstride + (size_t)y * out_pitch + x;
        if (vec && x + 4 <= cols) {
            const float4 v = *reinterpret_cast<const float4*>(i);
            *reinterpret_cast<uint2*>(o) = make_uint2(depth_u16(v.x) | depth_u16(v.y) << 16, depth_u16(v.z) | depth_u16(v.w) << 16);
        } else {
            for (int c = 0; c < 4 && x + c < cols; ++c) o[c] = (uint16_t)depth_u16(i[c]);
        }
    }
}

__global__ void k_q8_zero_counters(FrameCounters* c, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { c[i] = FrameCounters{}; c[i].path = 1; }
}

__global__ void k_q8_write_stats(const FrameCounters* __restrict__ c, int32_t* __restrict__ stats, int32_t* __restrict__ flags, int n, int path_code) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (stats) {
        stats[4 * i + 0] = c[i].extra_passes + 1;
        stats[4 * i + 1] = c[i].holes_after_first_fill;
        stats[4 * i + 2] = c[i].holes_after_extrapolation;
        stats[4 * i + 3] = c[i].needs_generic ? -1 : path_code;
    }
    if (flags) flags[i] = c[i].needs_generic;
}

}  // namespace

#ifndef DCMT_EMU
static cudaError_t tma_encode_3d(TensorMap3D* m, CUtensorMapDataType type, const void* base, int cols, int rows, int frames,
                                 size_t row_bytes, size_t frame_bytes, int box_cols, int box_rows) {
    typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                 const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                 CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static const EncodeFn fn = [] {
        void* f = nullptr;
        cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) f = nullptr;
        return reinterpret_cast<EncodeFn>(f);
    }();
    if (!fn || box_cols > 256 || box_rows > 256 || (row_bytes & 15) || (frame_bytes & 15) || (reinterpret_cast<uintptr_t>(base) & 15))
        return cudaErrorNotSupported;
    const cuuint64_t dims[3] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)frames};
    const cuuint64_t strides[2] = {(cuuint64_t)row_bytes, (cuuint64_t)frame_bytes};
    const cuuint32_t box[3] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows, 1u};
    const cuuint32_t estr[3] = {1u, 1u, 1u};
    const CUresult r = fn(m, type, 3, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                          CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? cudaSuccess : cudaErrorInvalidValue;
}
cudaError_t tma_encode_u16_3d(TensorMap3D* m, const uint16_t* base, int cols, int rows, int frames, size_t row_bytes,
                              size_t frame_bytes, int box_cols, int box_rows) {
    return tma_encode_3d(m, CU_TENSOR_MAP_DATA_TYPE_UINT16, base, cols, rows, frames, row_bytes, frame_bytes, box_cols, box_rows);
}
cudaError_t tma_encode_f32_3d(TensorMap3D* m, const float* base, int cols, int rows, int frames, size_t row_bytes,
                              size_t frame_bytes, int box_cols, int box_rows) {
    return tma_encode_3d(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, base, cols, rows, frames, row_bytes, frame_bytes, box_cols, box_rows);
}
#endif

// DCMT_NO_TMA=1: the front and the tail load their tiles with per-thread copies (the path for inputs a tensor map cannot
// describe), e.g. to test that path on any input
static bool tma_disabled() {
    static const bool no_tma = [] { const char* e = getenv("DCMT_NO_TMA"); return e && e[0] == '1'; }();
    return no_tma;
}

size_t q8_front_smem(int th, int tw) {
    // two region planes, the core-sized D plane, one quad of padding in front of / behind the region planes
    return ((size_t)2 * (th + FU + FD) * (tw / 8 + FLQ + FRQ) * 4 + (size_t)th * (tw / 8) * 4 + 8) * sizeof(uint32_t);
}

size_t q8_tail_smem(int th, int tw) {
    const size_t rowb = (size_t)(tw / 8 + 2 * TQ) * 4 * sizeof(uint32_t);
    return (size_t)2 * (th + 2 * TV) * rowb + (size_t)kListCap * sizeof(uint16_t);
}

void q8_choose_tile(int rows, int cols, int* th, int* tw) {
    // Tiles of at most 96 x 160 that divide the frame evenly (KITTI 352 x 1216 -> 88 x 152, 4 x 8 tiles).  Among the
    // splits near that size, take the one with the least halo work whose shared memory lets TWO CTAs of each kernel
    // share an SM (228 KB per SM, 1 KB reserved per CTA): the phases of the two overlap.
    static const int max_h = [] { const char* e = getenv("DCMT_TILE_MAX_H"); return e ? atoi(e) : 96; }();  // experiments
    const int ny0 = (rows + max_h - 1) / max_h, nx0 = (cols + 159) / 160;
    long best_cost = -1;
    for (int ny = ny0; ny <= ny0 + 3; ++ny)
        for (int nx = nx0; nx <= nx0 + 3; ++nx) {
            const int h = (rows + ny - 1) / ny, w = (((cols + nx - 1) / nx) + 7) / 8 * 8;
            if (h < 1 || w < 8) continue;
            const bool two = 2 * (q8_tail_smem(h, w) + 2048) <= 233472 && 2 * (q8_front_smem(h, w) + 2048) <= 233472;
            if (!two) continue;
            const long cost = (long)(h + 2 * TV) * (w + 16 * TQ) * ny * nx;
            if (best_cost < 0 || cost < best_cost) { best_cost = cost; *th = h; *tw = w; }
        }
    if (best_cost < 0) {  // cannot happen for the bounds above; keep the plain split
        *th = (rows + ny0 - 1) / ny0;
        *tw = (((cols + nx0 - 1) / nx0) + 7) / 8 * 8;
    }
}

cudaError_t q8_configure() {
    cudaError_t e = cudaFuncSetAttribute(k_q8_front<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(k_q8_front<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(k_q8_guided_front<true, GTL>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(k_q8_guided_front<false, GTW>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(k_q8_tail<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(k_q8_tail<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(k_q8_tail<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
}

cudaError_t q8_run_front(const Q8Plan& plan, const float* in, const uint16_t* in16, size_t in_pitch, size_t in_fstride, int n_frames,
                         int validate, cudaStream_t st) {
    // The front's tiles need not be the tail's (they meet in the global intermediate plane).  k_q8_front is latency bound
    // (its global loads, seven barriers), so DCMT_FRONT_CTAS CTAs per SM on lower tiles beat two tall ones although the
    // halo rows weigh more: the tallest even split of the rows whose shared memory fits that many CTAs.  Its width: the
    // kernel is bound by shared-memory bandwidth, and a quarter of its wavefronts were bank conflicts of warps that straddle
    // two rows of the region (rows of 21 quads, 42 half-quads: the second row starts on the banks the first one ends on).
    // A tile width of 8 (8 m - 2) pixels makes those rows 16 m half-quads long -- whole 128-byte wavefronts -- which is
    // worth 6 - 7 % at equal work (measured at 1216 x 352: 112-pixel tiles 1.387 ms against 1.480 ms for the tail's 152): such
    // widths compete with the tail's on (region quads x region rows), with that bonus.
    // DCMT_FRONT_TILE_H / DCMT_FRONT_TILE_W override the height bound / the width (experiments).
    static const int front_h = [] { const char* e = getenv("DCMT_FRONT_TILE_H"); const int v = e ? atoi(e) : 0; return v > 0 && v < 8 ? 8 : v; }();
    static const int front_w = [] { const char* e = getenv("DCMT_FRONT_TILE_W"); return e ? atoi(e) / 8 * 8 : -1; }();
    Q8Plan p = plan;
    auto height_for = [&](int tw) {
        int hmax = front_h > 0 ? front_h : plan.th;
        if (front_h <= 0 && DCMT_FRONT_CTAS > 2)
            while (hmax > 8 && (size_t)DCMT_FRONT_CTAS * (q8_front_smem(hmax, tw) + 1024) > (size_t)228 * 1024) --hmax;
        if (hmax >= plan.th) return plan.th;
        const int ny = (p.rows + hmax - 1) / hmax;
        return (p.rows + ny - 1) / ny;
    };
    auto width_ok = [&](int tw) { return tw >= 8 && (tw / 8 + FLQ + FRQ) * 9 <= QT; };  // more than 8 rows per sweep: col_pass relies on it
    if (front_w >= 0) {
        if (width_ok(front_w)) p.tw = front_w;
    } else {
        double best = -1.0;
        const int widths[4] = {plan.tw, 48, 112, 176};
        for (int tw : widths) {
            if (!width_ok(tw)) continue;
            const int th = height_for(tw), nx = (p.cols + tw - 1) / tw, ny = (p.rows + th - 1) / th;
            const double work = (double)nx * (tw / 8 + FLQ + FRQ) * ny * (th + FU + FD);
            const double cost = work * ((tw / 8 + FLQ + FRQ - 1) % 8 == 0 ? 0.93 : 1.0);
            if (best < 0 || cost < best) { best = cost; p.tw = tw; }
        }
    }
    p.th = height_for(p.tw);
    const size_t ncol = (size_t)p.mid_pitch * n_frames;
    DCMT_LAUNCH(k_q8_init_cols, dim3((unsigned)((ncol + 255) / 256)), dim3(256), 0, st, p.col_first, p.col_last, ncol,
                p.counters_ready ? nullptr : p.ctr, n_frames);
    // 16-byte vector loads need 16-byte aligned rows: 4 floats or 8 uint16 per unit
    const size_t unit = in16 ? 8 : 4;
    const uintptr_t base = in16 ? reinterpret_cast<uintptr_t>(in16) : reinterpret_cast<uintptr_t>(in);
    FrontArgs a{in, in16, in_pitch, in_fstride, p.mid, (size_t)p.mid_pitch, (size_t)p.mid_pitch * p.rows, p.col_first, p.col_last,
                p.ctr, p.rows, p.cols, p.th, p.tw, (int)(in_pitch % unit == 0 && in_fstride % unit == 0 && (base & 15) == 0), validate,
                make_colmap(p.tw / 8 + FLQ + FRQ, QT), make_colmap(p.tw / 8 + FLQ + FRQ - 1, QT), make_colmap(p.tw / 8, QT),
                make_items(2 * (p.tw / 8 + FLQ + FRQ - 1), QT), p.prof_front};
    a.codes = p.codes_in;
    // region load by TMA: a 3-D map (columns, rows, frames) of this chunk's input with the region as its box, unless the
    // input's layout cannot be mapped or a thread would hold more than kStagedSweeps quads of the staged region
    TensorMap3D tmap{};
    const int RH = p.th + FU + FD, RQ = p.tw / 8 + FLQ + FRQ;
    if (!tma_disabled() && RH <= kStagedSweeps * (QT / RQ)) {
        const cudaError_t e = in16 ? tma_encode_u16_3d(&tmap, in16, p.cols, p.rows, n_frames, in_pitch * 2, in_fstride * 2, RQ * 8, RH)
                                   : tma_encode_f32_3d(&tmap, in, p.cols, p.rows, n_frames, in_pitch * 4, in_fstride * 4, RQ * 8, RH);
        a.use_tma = e == cudaSuccess;
    }
    const dim3 grid((p.cols + p.tw - 1) / p.tw, (p.rows + p.th - 1) / p.th, n_frames);
    if (p.cols % 8 != 0) DCMT_LAUNCH(k_q8_front<true>, grid, dim3(QT), q8_front_smem(p.th, p.tw), st, a, tmap);
    else DCMT_LAUNCH(k_q8_front<false>, grid, dim3(QT), q8_front_smem(p.th, p.tw), st, a, tmap);
    return cudaGetLastError();
}

size_t q8_guided_smem(int th, int tw) { return ((size_t)3 * (th + FU + FD) * (tw / 8 + FLQ + FRQ) * 4 + 12) * sizeof(uint32_t) + sizeof(LabelTable); }

// tile height of the guided front: the tail's, or -- DCMT_GUIDED_CTAS > 1 -- the tallest even split of the rows whose shared
// memory lets that many CTAs share an SM (DCMT_GUIDED_TILE_H overrides the bound: experiments)
static int q8_guided_tile_h(int rows, int th, int tw) {
    static const int env_h = [] { const char* e = getenv("DCMT_GUIDED_TILE_H"); const int v = e ? atoi(e) : 0; return v > 0 && v < 8 ? 8 : v; }();
    int hmax = env_h > 0 ? env_h : th;
    if (env_h <= 0 && DCMT_GUIDED_CTAS > 1)
        while (hmax > 8 && (size_t)DCMT_GUIDED_CTAS * (q8_guided_smem(hmax, tw) + 1024) > (size_t)228 * 1024) --hmax;
    if (hmax >= th) return th;
    const int ny = (rows + hmax - 1) / hmax;
    return (rows + ny - 1) / ny;
}

size_t q8_guided_tile_flags(int rows, int cols, int th, int tw, int n_frames) {
    th = q8_guided_tile_h(rows, th, tw);
    return (size_t)((cols + tw - 1) / tw) * ((rows + th - 1) / th) * n_frames;
}

cudaError_t q8_run_guided_front(const Q8Plan& plan, const float* in, const uint16_t* in16, size_t in_pitch, size_t in_fstride,
                                const int32_t* labels, int n_clusters, int n_frames, int validate, int* tile_flags, cudaStream_t st) {
    Q8Plan p = plan;
    // DCMT_GUIDED_TILE_W: another tile width for the guided front (experiments; same bound as the plain front's)
    static const int guided_w = [] { const char* e = getenv("DCMT_GUIDED_TILE_W"); return e ? atoi(e) / 8 * 8 : 0; }();
    if (guided_w >= 8 && (guided_w / 8 + FLQ + FRQ) * 9 <= (GTL < GTW ? GTL : GTW)) p.tw = guided_w;
    p.th = q8_guided_tile_h(p.rows, p.th, p.tw);  // its own tiles: the kernels meet in the global intermediate plane
    const size_t ncol = (size_t)p.mid_pitch * n_frames;
    DCMT_LAUNCH(k_q8_init_cols, dim3((unsigned)((ncol + 255) / 256)), dim3(256), 0, st, p.col_first, p.col_last, ncol,
                p.counters_ready ? nullptr : p.ctr, n_frames);
    const size_t unit = in16 ? 8 : 4;
    const uintptr_t base = in16 ? reinterpret_cast<uintptr_t>(in16) : reinterpret_cast<uintptr_t>(in);
    const int RQ = p.tw / 8 + FLQ + FRQ;
    static const int guided_per_label = [] { const char* e = getenv("DCMT_GUIDED_PER_LABEL"); return e ? atoi(e) : 1; }();
    const dim3 grid((p.cols + p.tw - 1) / p.tw, (p.rows + p.th - 1) / p.th, n_frames);
    const size_t n_tiles = (size_t)grid.x * grid.y * n_frames;
    cudaError_t e = cudaMemsetAsync(tile_flags, 0, n_tiles * sizeof(int), st);
    if (e != cudaSuccess) return e;
    // column maps / magic reciprocals per thread count: load by region quads; items of the guided stage and of the vertical
    // pass by tw / 2 + 4 words (m_core), of the final pass by core quads (m_pass), label plane by region words (i_half)
    auto args = [&](int nt) {
        GuidedArgs g = GuidedArgs{FrontArgs{in, in16, in_pitch, in_fstride, p.mid, (size_t)p.mid_pitch, (size_t)p.mid_pitch * p.rows, p.col_first,
                                    p.col_last, p.ctr, p.rows, p.cols, p.th, p.tw,
                                    (int)(in_pitch % unit == 0 && in_fstride % unit == 0 && (base & 15) == 0), validate, make_colmap(RQ, nt),
                                    make_colmap(p.tw / 8, nt), make_colmap(p.tw / 2 + 4, nt), make_items(RQ * 4, nt), nullptr},
                          labels, n_clusters, guided_per_label, tile_flags};
        g.f.codes = p.codes_in;
        return g;
    };
    if (guided_per_label) DCMT_LAUNCH((k_q8_guided_front<true, GTL>), grid, dim3(GTL), q8_guided_smem(p.th, p.tw), st, args(GTL));
    // tiles the per-label kernel could not take (more distinct labels than its table holds) -- or all of them
    DCMT_LAUNCH((k_q8_guided_front<false, GTW>), grid, dim3(GTW), q8_guided_smem(p.th, p.tw) - sizeof(LabelTable), st, args(GTW));
    return cudaGetLastError();
}

cudaError_t q8_run_tail(const Q8Plan& p, float* out, uint16_t* out16, size_t out_pitch, size_t out_fstride, int n_frames, int blur,
                        cudaStream_t st) {
    // 4-pixel stores (16 bytes of float32 / 8 bytes of uint16) need every row start aligned to their size
    const int vec2 = out_pitch % 4 == 0 && out_fstride % 4 == 0 &&
                     (out16 ? (reinterpret_cast<uintptr_t>(out16) & 7) : (reinterpret_cast<uintptr_t>(out) & 15)) == 0;
    const int RQ = p.tw / 8 + 2 * TQ, RH = p.th + 2 * TV, SQ = p.tw / 8 + 2, MI = (p.tw / 2 + 2 + 3) / 4, NP = p.tw / 4;
    // shared-work median: word columns x runs of an even number of rows.  A run starts with four extra row sorts and a pair
    // merge, so longer runs execute fewer instructions while shorter ones keep more threads busy; measured on the B200 at the
    // KITTI tile (92 median rows x 78 word columns): runs of 16 / 20 / 28 / 32 / 36 / 40 rows -> tail 2.108 / 2.175 / 2.091 /
    // 2.070 / 2.136 / 2.223 ms per 1024 frames.  Hence: runs of about 32 rows, but at least ~200 items per CTA.
    const int NW = p.tw / 2 + 2, MH = p.th + 4;
    const int max_segs = QTT / NW > 0 ? QTT / NW : 1;
    int segs = (MH + 16) / 32;
    if (segs * NW < 200) segs = (200 + NW - 1) / NW;
    if (segs > max_segs) segs = max_segs;
    if (segs < 1) segs = 1;
    int med_len = 2 * ((MH + 2 * segs - 1) / (2 * segs));
    if (med_len < 8) med_len = 8;
    static const int env_len = [] { const char* e = getenv("DCMT_MED_LEN"); return e ? atoi(e) : 0; }();  // experiments
    if (env_len >= 2) med_len = env_len & ~1;
    const int med_segs = (MH + med_len - 1) / med_len;
    // tile load by TMA: a 3-D map (columns, rows, slots) of the intermediate plane whose column extent is the true
    // image width, so that the padding columns of the plane read as absent like everything else outside the image
    TensorMap3D tmap{};
    const int use_tma = !tma_disabled() && tma_encode_u16_3d(&tmap, p.mid, p.cols, p.rows, p.max_frames, (size_t)p.mid_pitch * 2,
                                                     (size_t)p.mid_pitch * p.rows * 2, RQ * 8, RH) == cudaSuccess;
    TailArgs a{p.mid, (size_t)p.mid_pitch, (size_t)p.mid_pitch * p.rows, p.col_first, p.col_last, p.ctr,
               out16 ? static_cast<void*>(out16) : static_cast<void*>(out), out_pitch,
               out_fstride, p.rows, p.cols, p.th, p.tw, blur, vec2, 1, use_tma,
               make_items(RQ, QTT), make_items(RQ * 4, QTT), make_items(SQ, QTT), make_items(SQ * 4, QTT), make_items(MI, QTT),
               make_items(NP, QTT), make_items(RQ * 2, QTT), make_items(NW, QTT), med_len, med_segs, p.lut ? kRankHundred : E_HUNDRED, p.lut, p.prof_tail};
    const dim3 grid((p.cols + p.tw - 1) / p.tw, (p.rows + p.th - 1) / p.th, n_frames);
    if (p.lut) DCMT_LAUNCH(k_q8_tail<true>, grid, dim3(QTT), q8_tail_smem(p.th, p.tw), st, a, tmap);
    else if (out16) DCMT_LAUNCH((k_q8_tail<false, true>), grid, dim3(QTT), q8_tail_smem(p.th, p.tw), st, a, tmap);
    else DCMT_LAUNCH(k_q8_tail<false>, grid, dim3(QTT), q8_tail_smem(p.th, p.tw), st, a, tmap);
    return cudaGetLastError();
}

cudaError_t q8_zero_counters(const Q8Plan& p, int n_frames, cudaStream_t st) {
    DCMT_LAUNCH(k_q8_zero_counters, dim3((n_frames + 127) / 128), dim3(128), 0, st, p.ctr, n_frames);
    return cudaGetLastError();
}

cudaError_t q8_write_stats(const Q8Plan& p, int32_t* stats, int32_t* flags, int n_frames, cudaStream_t st) {
    DCMT_LAUNCH(k_q8_write_stats, dim3((n_frames + 127) / 128), dim3(128), 0, st, p.ctr, stats, flags, n_frames, p.lut ? 2 : 1);
    return cudaGetLastError();
}

cudaError_t q8_convert_u16(const uint16_t* in, size_t in_pitch, size_t in_fstride, float* out, int rows, int cols, int n_frames,
                           cudaStream_t st) {
    DCMT_LAUNCH(k_u16_to_f32, dim3((cols + 255) / 256, rows, n_frames), dim3(256), 0, st, in, in_pitch, in_fstride, out, rows, cols);
    return cudaGetLastError();
}

cudaError_t depth_to_u16(const float* in, size_t in_pitch, size_t in_fstride, uint16_t* out, size_t out_pitch, size_t out_fstride,
                         int rows, int cols, int n_frames, cudaStream_t st) {
    const int vec = in_pitch % 4 == 0 && in_fstride % 4 == 0 && (reinterpret_cast<uintptr_t>(in) & 15) == 0 && out_pitch % 4 == 0 &&
                    out_fstride % 4 == 0 && (reinterpret_cast<uintptr_t>(out) & 7) == 0;
    const unsigned gx = (unsigned)((cols + 1023) / 1024), gy = (unsigned)(rows < 65535 ? rows : 65535);
    for (int f0 = 0; f0 < n_frames; f0 += 65535) {  // grid z limit
        const int nf = n_frames - f0 < 65535 ? n_frames - f0 : 65535;
        DCMT_LAUNCH(k_depth_to_u16, dim3(gx, gy, nf), dim3(256), 0, st, in + (size_t)f0 * in_fstride, in_pitch, in_fstride,
                    out + (size_t)f0 * out_fstride, out_pitch, out_fstride, rows, cols, vec);
        const cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

cudaError_t q8_decode_plane(const uint16_t* mid, size_t mid_pitch, float* out, int rows, int cols, cudaStream_t st) {
    DCMT_LAUNCH(k_q8_decode, dim3((cols + 127) / 128, rows), dim3(128), 0, st, mid, mid_pitch, out, rows, cols);
    return cudaGetLastError();
}

}  // namespace dcmt
