// api.cu -- the C ABI of libdcmt.so (include/dcmt.h): argument validation, workspace cache,
// chunking, path selection.  No compute happens on the host and there is no CPU fallback.
#include "../../include/dcmt.h"

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <map>
#include <mutex>
#include <utility>
#include <vector>
#include <algorithm>

#include "common.cuh"
#include "evaluate.cuh"
#include "fused_q8.cuh"
#include "generic.cuh"
#include "project.cuh"
#include "rank_f32.cuh"
#include "color.cuh"
#include "slic.cuh"
#include "stereo.cuh"

#include <atomic>

namespace dcmt {
static std::atomic<long long> g_launches{0};
void note_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
}  // namespace dcmt

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

int cuda_fail(cudaError_t e, const char* what) {
    return fail(DCMT_E_CUDA, "%s: %s", what, cudaGetErrorString(e));
}

// DCMT_OK, or the error of a launch or copy that returned `e`
int cuda_rc(cudaError_t e, const char* what) { return e == cudaSuccess ? DCMT_OK : cuda_fail(e, what); }

#define API_CUDA(x, what)                                  \
    do {                                                   \
        cudaError_t e__ = (x);                             \
        if (e__ != cudaSuccess) return cuda_fail(e__, what); \
    } while (0)

// ---- workspace cache: one grow-only device arena per (device, stream) ----
struct Arena {
    char* base = nullptr;
    size_t cap = 0, used = 0;
    bool overflow = false;  // a carve() went past cap since the last acquire: the caller must not launch anything
    bool counting = false;  // sizes a workspace: carve() adds up what it takes and hands out no memory (acquire_carved)
};
std::mutex g_mu;
std::map<std::pair<int, cudaStream_t>, Arena> g_arenas;

int arena_acquire(cudaStream_t st, size_t bytes, Arena** out) {
    int dev = 0;
    API_CUDA(cudaGetDevice(&dev), "cudaGetDevice");
    std::lock_guard<std::mutex> lk(g_mu);
    Arena& a = g_arenas[{dev, st}];
    if (a.cap < bytes) {
        if (a.base) {
            // work enqueued earlier on this stream may still use the old block
            API_CUDA(cudaStreamSynchronize(st), "cudaStreamSynchronize");
            cudaFree(a.base);
            a.base = nullptr;
            a.cap = 0;
        }
        void* p = nullptr;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess) return fail(DCMT_E_NOMEM, "workspace of %zu bytes: %s", bytes, cudaGetErrorString(e));
        a.base = static_cast<char*>(p);
        a.cap = bytes;
    }
    a.used = 0;
    a.overflow = false;
    *out = &a;
    return DCMT_OK;
}

// Bounds-checked: a request past the end of the arena sets `overflow` and returns the arena base (valid memory that
// must not be used); acquire_carved checks it before anything is launched.
template <class T>
T* carve(Arena* a, size_t count) {
    const size_t bytes = (count * sizeof(T) + 255) & ~size_t(255);
    if (a->counting) {
        a->used += bytes;
        return nullptr;
    }
    if (a->used + bytes > a->cap) {
        a->overflow = true;
        return reinterpret_cast<T*>(a->base);
    }
    T* p = reinterpret_cast<T*>(a->base + a->used);
    a->used += bytes;
    return p;
}

// The workspace of one step of a call, in the arena of `st`: carve_ws(Arena*) runs once on a counting arena to size it, then
// on the stream's arena for real.  The size comes from the code that lays the workspace out, so the two cannot disagree.
template <class Carve>
int acquire_carved(cudaStream_t st, Carve&& carve_ws) {
    Arena count, *ar = nullptr;
    count.counting = true;
    carve_ws(&count);
    if (int rc = arena_acquire(st, count.used, &ar)) return rc;
    carve_ws(ar);
    return ar->overflow ? fail(DCMT_E_NOMEM, "internal: workspace arena of %zu bytes is too small for this call", ar->cap) : DCMT_OK;
}

long env_long(const char* name) {
    const char* s = getenv(name);
    return s ? atol(s) : 0L;
}

// Frames per chunk: as many as a pixel budget allows (DCMT_FUSED_CHUNK / DCMT_GENERIC_CHUNK override it with a frame
// count), split evenly.
// - fused path, 2^28 pixels (627 KITTI frames; about 0.5 GB of uint16 intermediate plus 2 GB of fix-up scratch).  Large
//   grids matter more than L2 residency of the intermediate plane: the kernels are issue-bound (DRAM a few per cent
//   busy), while every launch ends in a partially filled wave (79-frame chunks: 8.5 waves per launch, 11 % slower end to
//   end than 512-frame chunks on the B200).
// - generic pipeline, 2^27 pixels (313 KITTI frames, 1 GB of float scratch).  Larger grids beat L2 residency of the two
//   float planes here as well (20-frame chunks were 10 % slower).
int chunk_frames(int rows, int cols, int n_frames, bool fused) {
    static const long fused_env = env_long("DCMT_FUSED_CHUNK"), generic_env = env_long("DCMT_GENERIC_CHUNK");
    const long env = fused ? fused_env : generic_env;
    long cap = env > 0 ? env : (long)(((size_t)1 << (fused ? 28 : 27)) / ((size_t)rows * cols));
    if (cap < 1) cap = 1;
    if (cap > 65535) cap = 65535;
    const long nchunks = (n_frames + cap - 1) / cap;
    long c = nchunks > 0 ? (n_frames + nchunks - 1) / nchunks : 1;
    if (c < 1) c = 1;
    return (int)c;
}

bool overlaps(const void* a, size_t an, const void* b, size_t bn) {
    const char* pa = static_cast<const char*>(a);
    const char* pb = static_cast<const char*>(b);
    return pa < pb + bn && pb < pa + an;
}

struct Geometry {
    size_t pitch, fstride;  // elements
    size_t span_bytes;      // bytes touched by the whole batch
};

int check_planes(int rows, int cols, int n_frames) {
    if (rows < 1 || cols < 1) return fail(DCMT_E_BADARG, "rows and cols must be >= 1 (got %d x %d)", rows, cols);
    if (n_frames < 0) return fail(DCMT_E_BADARG, "n_frames must be >= 0 (got %d)", n_frames);
    return DCMT_OK;
}

int check_geometry(int rows, int cols, size_t pitch_bytes, size_t frame_stride_bytes, int n_frames, Geometry* g,
                   size_t elem = sizeof(float)) {
    if (int rc = check_planes(rows, cols, n_frames)) return rc;
    if ((size_t)rows * (size_t)cols > (size_t)1 << 30) return fail(DCMT_E_UNSUPPORTED, "frame larger than 2^30 pixels");
    if (pitch_bytes == 0) pitch_bytes = (size_t)cols * elem;
    if (pitch_bytes % elem != 0 || pitch_bytes < (size_t)cols * elem)
        return fail(DCMT_E_BADARG, "pitch_bytes %zu invalid for %d columns of %zu bytes", pitch_bytes, cols, elem);
    if (frame_stride_bytes == 0) frame_stride_bytes = pitch_bytes * rows;
    if (frame_stride_bytes % elem != 0 || frame_stride_bytes < pitch_bytes * (size_t)(rows - 1) + (size_t)cols * elem)
        return fail(DCMT_E_BADARG, "frame_stride_bytes %zu invalid", frame_stride_bytes);
    g->pitch = pitch_bytes / elem;
    g->fstride = frame_stride_bytes / elem;
    g->span_bytes = n_frames ? frame_stride_bytes * (size_t)(n_frames - 1) + pitch_bytes * (size_t)(rows - 1) + (size_t)cols * elem : 0;
    return DCMT_OK;
}

int check_device() {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n < 1)
        return fail(DCMT_E_CUDA, "no CUDA device available (%s); libdcmt has no CPU fallback",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
    return DCMT_OK;
}

// ---- optional per-kernel timing of the fused path (dcmt_profile_begin / dcmt_profile_end): CUDA events recorded on
// the launch stream around k_q8_front and k_q8_tail of every chunk, read back when profiling ends
struct ProfEvents {
    cudaEvent_t e[3];
};
bool g_prof_on = false;
std::vector<ProfEvents> g_prof_events;

cudaError_t prof_mark(cudaStream_t st, int which, ProfEvents* pe) {
    if (!g_prof_on) return cudaSuccess;
    cudaError_t e = cudaEventCreate(&pe->e[which]);
    if (e != cudaSuccess) return e;
    return cudaEventRecord(pe->e[which], st);
}

// cv::cvtColor(COLOR_BGR2Lab) + Slic::generate_superpixels in front of a guided completion: the labels are made on the
// device from the caller's BGR frames (dcmt_interpolate_with_superpixels_bgr_*) instead of being passed in
struct BgrFront {
    const uint8_t* bgr;
    size_t pitch, fstride;  // bytes; the ABI's 0 = dense until validate_completion fills them in
    int step, nc, iterations;
};

// one completion call as its entry point describes it (checked by validate_completion)
struct CompletionCall {
    const int32_t* labels;
    int n_clusters;
    bool guided;
    int rows, cols, blur, flags;
    BgrFront* front = nullptr;  // labels from BGR frames (`labels` unused; validate_completion sets n_clusters)
};

// the strict-q8 fused path serves plain img_completion with blur none/gaussian on frames of a sane size
bool fused_applies(const CompletionCall& cc) {
    if (cc.flags == DCMT_PATH_GENERIC || cc.blur == DCMT_BLUR_BILATERAL) return false;
    if (cc.guided && (cc.n_clusters < 0 || cc.n_clusters > 65535)) return false;  // the fused guided front keeps labels as uint16
    if (cc.rows < dcmt::kQ8MinRows || cc.cols < dcmt::kQ8MinCols || cc.rows > dcmt::kQ8MaxRows) return false;
    int th, tw;
    dcmt::q8_choose_tile(cc.rows, cc.cols, &th, &tw);
    return dcmt::q8_tail_smem(th, tw) <= 200 * 1024 && dcmt::q8_front_smem(th, tw) <= 200 * 1024 &&
           (!cc.guided || dcmt::q8_guided_smem(th, tw) <= 200 * 1024);
}

// One side of a completion call: float32 metres (`f`) or KITTI uint16, metres * 256 (`u`; main.cpp:75-82 on the way in,
// the rule of dcmt_depth_to_u16 on the way out).  Pitch and frame stride are in elements; the entry points fill in the
// ABI's bytes (0 = packed), which validate_completion checks and converts.
struct InDesc {
    const float* f = nullptr;
    const uint16_t* u = nullptr;
    size_t pitch = 0, fstride = 0;
    size_t elem() const { return u ? sizeof(uint16_t) : sizeof(float); }
    const void* ptr() const { return u ? static_cast<const void*>(u) : f; }
    InDesc frames_from(size_t f0) const {
        InDesc o = *this;
        if (u) o.u += f0 * fstride;
        else o.f += f0 * fstride;
        return o;
    }
};

struct OutDesc {
    float* f = nullptr;
    uint16_t* u = nullptr;
    size_t pitch = 0, fstride = 0;
    size_t elem() const { return u ? sizeof(uint16_t) : sizeof(float); }
    void* ptr() const { return u ? static_cast<void*>(u) : f; }
    OutDesc frames_from(size_t f0) const {
        OutDesc o = *this;
        if (u) o.u += f0 * fstride;
        else o.f += f0 * fstride;
        return o;
    }
};

// The generic pipeline's scratch for launches of up to `chunk` frames, in the workspace fields of a GenericChunk: two float
// planes, the per-frame counters and, for the bilateral blur, its min / max words and range LUTs.  The fused path shares
// the planes and counters (fix-ups).
dcmt::GenericChunk carve_generic(Arena* ar, int rows, int cols, int chunk, bool bilateral) {
    const size_t px = (size_t)rows * cols * chunk;
    dcmt::GenericChunk g{};
    g.w1 = carve<float>(ar, px);
    g.w2 = carve<float>(ar, px);
    g.ctr = carve<dcmt::FrameCounters>(ar, chunk);
    g.minmax = bilateral ? carve<unsigned>(ar, 2 * (size_t)chunk) : nullptr;
    g.lut = bilateral ? carve<float>(ar, dcmt::generic_lut_floats() * chunk) : nullptr;
    return g;
}

// The fused path's buffers for launches of up to `chunk` frames, next to the generic scratch `g`: the uint16 intermediate
// plane and its column keys, the tile flags of the guided front and -- on DCMT_PATH_RANK -- the per-frame dictionary, its
// sizes and the code plane (rank_f32.cu).
struct FusedWork {
    dcmt::Q8Plan p{};
    int* tile_flags = nullptr;
    float* lut = nullptr;
    int* lut_count = nullptr;
    uint16_t* codes = nullptr;
};

size_t pad8(int cols) { return ((size_t)cols + 7) / 8 * 8; }

FusedWork carve_fused(Arena* ar, int rows, int cols, int chunk, bool guided, bool rank, const dcmt::GenericChunk& g) {
    FusedWork w;
    dcmt::Q8Plan& p = w.p;
    p.rows = rows;
    p.cols = cols;
    dcmt::q8_choose_tile(rows, cols, &p.th, &p.tw);
    p.mid_pitch = (int)pad8(cols);
    p.max_frames = chunk;
    p.mid = carve<uint16_t>(ar, (size_t)rows * p.mid_pitch * chunk);
    p.col_first = carve<uint32_t>(ar, (size_t)p.mid_pitch * chunk);
    p.col_last = carve<uint32_t>(ar, (size_t)p.mid_pitch * chunk);
    p.ctr = g.ctr;
    p.w1 = g.w1;
    p.w2 = g.w2;
    if (guided) w.tile_flags = carve<int>(ar, dcmt::q8_guided_tile_flags(rows, cols, p.th, p.tw, chunk));
    if (rank) {
        w.lut = carve<float>(ar, (size_t)dcmt::kRankMaxValid * chunk);
        w.lut_count = carve<int>(ar, (size_t)chunk);
        w.codes = carve<uint16_t>(ar, (size_t)rows * p.mid_pitch * chunk);
        p.codes_in = 1;
        p.counters_ready = 1;
        p.lut = w.lut;
    }
    return w;
}

// The workspace of a completion pass over up to `frames` frames, in launches of up to `chunk` frames: the generic scratch,
// then the fused path's buffers or -- the generic pipeline reads and writes float32 -- a plane in front of it for uint16
// input and one behind it for uint16 output.
struct CompletionWork {
    bool fused;
    int chunk;
    dcmt::GenericChunk g;
    FusedWork f;
    float *conv, *staged;
};

CompletionWork carve_completion(Arena* ar, const CompletionCall& cc, int frames, bool u16_in, bool u16_out) {
    CompletionWork w{};
    w.fused = fused_applies(cc);
    w.chunk = chunk_frames(cc.rows, cc.cols, frames, w.fused);
    w.g = carve_generic(ar, cc.rows, cc.cols, w.chunk, cc.blur == DCMT_BLUR_BILATERAL);
    const size_t px = (size_t)cc.rows * cc.cols * w.chunk;
    if (w.fused) w.f = carve_fused(ar, cc.rows, cc.cols, w.chunk, cc.guided, cc.flags == DCMT_PATH_RANK, w.g);
    w.conv = !w.fused && u16_in ? carve<float>(ar, px) : nullptr;
    w.staged = !w.fused && u16_out ? carve<float>(ar, px) : nullptr;
    return w;
}

// Whether a completion pass reports the frames it did not serve ("not served" flags): float32 input on the fused kernels,
// except in the debugging calls (copy only, per-stage planes)
bool writes_flags(const CompletionCall& cc, bool f32_in, bool debug) { return fused_applies(cc) && f32_in && !debug; }

// The level that redoes the frames a pass at `level` did not serve: strict-q8 kernels -> dictionary (rank_f32.cu) ->
// generic pipeline; -1 below DCMT_PATH_GENERIC and DCMT_PATH_FUSED
int path_below(int level) {
    return level == DCMT_PATH_AUTO ? DCMT_PATH_RANK : level == DCMT_PATH_RANK ? DCMT_PATH_GENERIC : -1;
}

// Enqueue n_frames through the pipeline on the workspace `w` (carve_completion for at least n_frames frames); every pointer
// is a device pointer.  Never synchronises.  On the fused path `redo_flags` (device, one int32 per frame, optional) receives
// 1 for frames that turned out not to be strict q8: their output is NOT valid and the caller must redo them one level down.
// `stages` (the per-stage planes of DCMT_PATH_GENERIC calls) and `stage_mask` are passed to the generic pipeline.
//
// uint16 input is strict q8 by construction (the drivers map every path but DCMT_PATH_GENERIC to DCMT_PATH_FUSED): the
// fused kernels read it directly and nothing is validated or redone; shapes the fused kernels do not serve get a
// convertTo(CV_32F, 1/256) (main.cpp:79) into a workspace plane in front of the generic pipeline.  uint16 output: the
// fused tail stores it directly; the generic pipeline writes a float workspace plane that depth_to_u16 converts.
int enqueue_completion(const CompletionCall& cc, const CompletionWork& w, const InDesc& in, const int32_t* labels, const OutDesc& out,
                       int n_frames, int32_t* stats, int32_t* redo_flags, float* stages, uint32_t* stage_mask, cudaStream_t st) {
    const int rows = cc.rows, cols = cc.cols;
    // launches never take more frames than the workspace holds, whatever chunk sizes the environment sets
    const int chunk = std::min(chunk_frames(rows, cols, n_frames, w.fused), w.chunk);
    const size_t fpix = (size_t)rows * cols;
    if (w.fused) {
        // DCMT_PATH_RANK: float32 frames through the per-frame dictionary (rank_f32.cu) in front of the same kernels
        const bool rank = cc.flags == DCMT_PATH_RANK;
        const FusedWork& fw = w.f;
        const dcmt::Q8Plan& p = fw.p;
        if (rank) API_CUDA(dcmt::rank_configure(), "kernel attribute setup");
        for (int f0 = 0; f0 < n_frames; f0 += chunk) {
            const int nf = n_frames - f0 < chunk ? n_frames - f0 : chunk;
            ProfEvents pe{};
            API_CUDA(prof_mark(st, 0, &pe), "profiling event");
            // the front reads the dictionary codes, the uint16 input, or the float32 input (validated unless DCMT_PATH_FUSED)
            InDesc fin = in.frames_from((size_t)f0);
            if (rank) {
                API_CUDA(dcmt::q8_zero_counters(p, nf, st), "counter setup launch");
                API_CUDA(dcmt::rank_build(fin.f, fin.pitch, fin.fstride, rows, cols, nf, fw.lut, fw.lut_count, fw.codes, (size_t)p.mid_pitch,
                                          p.ctr, st),
                         "dictionary launch");
                fin = InDesc{nullptr, fw.codes, (size_t)p.mid_pitch, (size_t)p.mid_pitch * rows};
            }
            const int validate = fin.f && cc.flags != DCMT_PATH_FUSED;
            if (cc.guided)
                API_CUDA(dcmt::q8_run_guided_front(p, fin.f, fin.u, fin.pitch, fin.fstride, labels + (size_t)f0 * fpix, cc.n_clusters, nf,
                                                   validate, fw.tile_flags, st),
                         "fused guided front launch");
            else
                API_CUDA(dcmt::q8_run_front(p, fin.f, fin.u, fin.pitch, fin.fstride, nf, validate, st), "fused front launch");
            API_CUDA(prof_mark(st, 1, &pe), "profiling event");
            const OutDesc o = out.frames_from((size_t)f0);
            API_CUDA(dcmt::q8_run_tail(p, o.f, o.u, o.pitch, o.fstride, nf, cc.blur, st), "fused tail launch");
            API_CUDA(prof_mark(st, 2, &pe), "profiling event");
            if (g_prof_on) {
                std::lock_guard<std::mutex> lk(g_mu);
                g_prof_events.push_back(pe);
            }
            if (stats || redo_flags)
                API_CUDA(dcmt::q8_write_stats(p, stats ? stats + (size_t)f0 * DCMT_STATS_STRIDE : nullptr,
                                              redo_flags ? redo_flags + f0 : nullptr, nf, st),
                         "stats launch");
        }
        return DCMT_OK;
    }
    for (int f0 = 0; f0 < n_frames; f0 += chunk) {
        const int nf = n_frames - f0 < chunk ? n_frames - f0 : chunk;
        const InDesc i = in.frames_from((size_t)f0);
        dcmt::GenericChunk c = w.g;
        if (w.conv) {
            API_CUDA(dcmt::q8_convert_u16(i.u, i.pitch, i.fstride, w.conv, rows, cols, nf, st), "uint16 conversion launch");
            c.in = w.conv;
            c.in_pitch = (size_t)cols;
            c.in_fstride = fpix;
        } else {
            c.in = i.f;
            c.in_pitch = i.pitch;
            c.in_fstride = i.fstride;
        }
        c.labels = cc.guided ? labels + (size_t)f0 * fpix : nullptr;
        c.n_clusters = cc.n_clusters;
        c.guided = cc.guided;
        const OutDesc o = out.frames_from((size_t)f0);
        c.out = w.staged ? w.staged : o.f;
        c.out_pitch = w.staged ? (size_t)cols : o.pitch;
        c.out_fstride = w.staged ? fpix : o.fstride;
        c.rows = rows;
        c.cols = cols;
        c.n_frames = nf;
        c.blur = cc.blur;
        c.stats = stats ? stats + (size_t)f0 * DCMT_STATS_STRIDE : nullptr;
        c.stages = stages;
        c.stage_mask = stage_mask;
        API_CUDA(dcmt::generic_run_chunk(c, st), "generic pipeline launch");
        if (w.staged)
            API_CUDA(dcmt::depth_to_u16(w.staged, (size_t)cols, fpix, o.u, o.pitch, o.fstride, rows, cols, nf, st), "uint16 conversion launch");
    }
    return DCMT_OK;
}

// pinned host scratch for the redo flags, one per (device, stream) like the arenas (grow-only): calls on different
// streams never share a buffer; calls on the SAME stream are ordered by the caller, and a buffer is only replaced
// after that stream has drained (the previous call's read-back may still be in flight otherwise).  The host-pointer
// entry points use the key (device, nullptr-stream of the host pipeline) under their per-device mutex.
struct PinnedFlags {
    int32_t* p = nullptr;
    size_t cap = 0;
};
std::map<std::pair<int, cudaStream_t>, PinnedFlags> g_pinned;

int pinned_flags(cudaStream_t key, size_t n, int32_t** out) {
    int dev = 0;
    API_CUDA(cudaGetDevice(&dev), "cudaGetDevice");
    std::lock_guard<std::mutex> lk(g_mu);
    PinnedFlags& pf = g_pinned[{dev, key}];
    if (pf.cap < n) {
        if (pf.p) {
            API_CUDA(cudaStreamSynchronize(key), "cudaStreamSynchronize");
            cudaFreeHost(pf.p);
        }
        pf.p = nullptr;
        pf.cap = 0;
        void* q = nullptr;
        cudaError_t e = cudaMallocHost(&q, n * sizeof(int32_t));
        if (e != cudaSuccess) return fail(DCMT_E_NOMEM, "pinned flag buffer: %s", cudaGetErrorString(e));
        pf.p = static_cast<int32_t*>(q);
        pf.cap = n;
    }
    *out = pf.p;
    return DCMT_OK;
}

// SLIC's own limits (slic.cpp:72-99 and the kernels' index arithmetic), on frames already checked to be 1..2^30 pixels
int check_slic(int rows, int cols, int step, int nc, int iterations) {
    if (nc == 0 || iterations < 0) return fail(DCMT_E_BADARG, "nc %d, iterations %d", nc, iterations);
    if (step < 4) return fail(DCMT_E_UNSUPPORTED, "step %d: find_local_minimum (slic.cpp:72-99) reads outside the image below 4", step);
    if (rows >= 1 << 24 || cols >= 1 << 24) return fail(DCMT_E_UNSUPPORTED, "SLIC frames are limited to 2^24 rows / columns");
    return DCMT_OK;
}

// The pitch and frame stride in bytes of n_frames BGR frames of rows x cols (0 = dense: filled in); *span receives the bytes
// the frames cover
int check_bgr_geometry(int rows, int cols, size_t* pitch, size_t* fstride, int n_frames, size_t* span) {
    const size_t row = (size_t)cols * 3;
    if (*pitch == 0) *pitch = row;
    if (*fstride == 0) *fstride = *pitch * rows;
    if (*pitch < row) return fail(DCMT_E_BADARG, "bgr_pitch_bytes %zu below %d columns of 3 bytes", *pitch, cols);
    const size_t frame = *pitch * (size_t)(rows - 1) + row;
    if (*fstride < frame) return fail(DCMT_E_BADARG, "bgr_frame_stride_bytes %zu invalid", *fstride);
    *span = n_frames ? *fstride * (size_t)(n_frames - 1) + frame : 0;
    return DCMT_OK;
}

// Checks a completion call -- pointers, labels, blur, flags, input geometry, output geometry, overlap, in this order, then
// for a BGR front its pointer, SLIC's arguments, its geometry and its overlap with the output -- and converts the pitches
// and frame strides of `in` and `out` from the ABI's bytes into elements.  A BGR front gets its dense pitch / frame stride
// filled in and `cc.n_clusters` is set to SLIC's centre count.
int validate_completion(CompletionCall& cc, InDesc* in, OutDesc* out, int n_frames) {
    if (!in->ptr() || !out->ptr()) return fail(DCMT_E_BADARG, "null image pointer");
    if (cc.guided && !cc.labels && !cc.front) return fail(DCMT_E_BADARG, "null label pointer");
    if (cc.blur < DCMT_BLUR_NONE || cc.blur > DCMT_BLUR_BILATERAL) return fail(DCMT_E_BADARG, "blur_type %d", cc.blur);
    if (cc.flags < DCMT_PATH_AUTO || cc.flags > DCMT_PATH_RANK) return fail(DCMT_E_BADARG, "flags %d", cc.flags);
    Geometry gi, go;
    int rc = check_geometry(cc.rows, cc.cols, in->pitch, in->fstride, n_frames, &gi, in->elem());
    if (rc) return rc;
    if ((rc = check_geometry(cc.rows, cc.cols, out->pitch, out->fstride, n_frames, &go, out->elem()))) return rc;
    if (n_frames && overlaps(in->ptr(), gi.span_bytes, out->ptr(), go.span_bytes)) return fail(DCMT_E_BADARG, "input and output overlap");
    if (BgrFront* fr = cc.front) {
        if (!fr->bgr) return fail(DCMT_E_BADARG, "null image pointer");
        if ((rc = check_slic(cc.rows, cc.cols, fr->step, fr->nc, fr->iterations))) return rc;
        size_t span = 0;
        if ((rc = check_bgr_geometry(cc.rows, cc.cols, &fr->pitch, &fr->fstride, n_frames, &span))) return rc;
        if (n_frames && overlaps(fr->bgr, span, out->ptr(), go.span_bytes)) return fail(DCMT_E_BADARG, "BGR input and output overlap");
        cc.n_clusters = dcmt::slic_center_count(cc.rows, cc.cols, fr->step);
    }
    in->pitch = gi.pitch;
    in->fstride = gi.fstride;
    out->pitch = go.pitch;
    out->fstride = go.fstride;
    return DCMT_OK;
}

// frames [f, e) of a call
struct Run {
    int f, e;
};

// the runs of consecutive frames whose flag is set, in frame order: the frames a pass did not serve
std::vector<Run> flagged_runs(const int32_t* flags, int n) {
    std::vector<Run> runs;
    for (int f = 0; f < n;) {
        if (!flags[f]) { ++f; continue; }
        int e = f;
        while (e < n && flags[e]) ++e;
        runs.push_back(Run{f, e});
        f = e;
    }
    return runs;
}

// uint16 input needs no validation: AUTO, RANK and FUSED are the same thing there
int input_path(const InDesc& in, int flags) { return in.u && flags != DCMT_PATH_GENERIC ? DCMT_PATH_FUSED : flags; }

// device-pointer driver of every completion entry point
int run_completion(CompletionCall cc, InDesc in, OutDesc out, int n_frames, int32_t* stats, cudaStream_t st, float* stages = nullptr,
                   uint32_t* stage_mask = nullptr) {
    int rc = validate_completion(cc, &in, &out, n_frames);
    if (rc) return rc;
    if (n_frames == 0) return DCMT_OK;
    if ((rc = check_device())) return rc;
    API_CUDA(dcmt::generic_configure(), "kernel attribute setup");
    API_CUDA(dcmt::q8_configure(), "kernel attribute setup");
    cc.flags = input_path(in, cc.flags);
    const bool flagged = writes_flags(cc, in.f, stages);
    int32_t* d_flags = nullptr;
    CompletionWork w;
    if ((rc = acquire_carved(st, [&](Arena* a) {
             d_flags = flagged ? carve<int32_t>(a, (size_t)n_frames) : nullptr;
             w = carve_completion(a, cc, n_frames, in.u, out.u);
         })))
        return rc;
    if ((rc = enqueue_completion(cc, w, in, cc.labels, out, n_frames, stats, d_flags, stages, stage_mask, st))) return rc;
    if (!flagged || path_below(cc.flags) < 0) return DCMT_OK;  // DCMT_PATH_FUSED: fully asynchronous, stats[3] = -1 marks bad frames
    // DCMT_PATH_AUTO / DCMT_PATH_RANK: read the per-frame "not served" flags back (one synchronisation per pass) and redo
    // those frames one level down
    int32_t* h_flags = nullptr;
    if ((rc = pinned_flags(st, (size_t)n_frames, &h_flags))) return rc;
    API_CUDA(cudaMemcpyAsync(h_flags, d_flags, (size_t)n_frames * sizeof(int32_t), cudaMemcpyDeviceToHost, st), "flag readback");
    API_CUDA(cudaStreamSynchronize(st), "kernel execution");
    for (cc.flags = path_below(cc.flags); cc.flags >= 0; cc.flags = path_below(cc.flags)) {
        const bool want_flags = writes_flags(cc, in.f, false);
        const std::vector<Run> runs = flagged_runs(h_flags, n_frames);
        if (runs.empty()) break;
        for (const Run& r : runs) {
            const int f = r.f, n = r.e - r.f;
            // the previous pass has completed (stream synchronised): the arena is free again, but this pass may need more (the
            // generic pipeline: two float planes per frame of its chunk)
            int32_t* run_flags = nullptr;
            if ((rc = acquire_carved(st, [&](Arena* a) {
                     run_flags = want_flags ? carve<int32_t>(a, (size_t)n) : nullptr;
                     w = carve_completion(a, cc, n, in.u, out.u);
                 })))
                return rc;
            if ((rc = enqueue_completion(cc, w, in.frames_from((size_t)f), cc.guided ? cc.labels + (size_t)f * cc.rows * cc.cols : nullptr,
                                         out.frames_from((size_t)f), n, stats ? stats + (size_t)f * DCMT_STATS_STRIDE : nullptr, run_flags,
                                         nullptr, nullptr, st)))
                return rc;
            if (want_flags) {
                // arenas are reused by the next run of this pass in stream order; the flags leave through the pinned buffer first
                API_CUDA(cudaMemcpyAsync(h_flags + f, run_flags, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, st), "flag readback");
                API_CUDA(cudaStreamSynchronize(st), "kernel execution");
            }
        }
    }
    return DCMT_OK;
}

// ---- SLIC on a workspace carved from an arena the caller holds, so that the chained calls keep their staging buffers,
// labels and completion workspace in the same arena: the work arrays of SlicWork for up to n frames and, with from_bgr,
// the Lab frames
struct SlicBuffers {
    dcmt::SlicWork w{};
    uint8_t* lab = nullptr;
};

SlicBuffers carve_slic(Arena* ar, int rows, int cols, int n, int step, bool from_bgr) {
    SlicBuffers s;
    const int k = dcmt::slic_center_count(rows, cols, step);
    const size_t nbins = dcmt::slic_bins(rows, cols, step, &s.w.bins_x, &s.w.bins_y);
    const size_t kk = (k > 0 ? (size_t)k : 1) * n, nb = nbins * n;
    s.w.centers = carve<double>(ar, kk * 5);
    s.w.sums = carve<unsigned long long>(ar, kk * 6);
    s.w.bin_count = carve<int>(ar, nb + n);
    s.w.bin_fill = carve<int>(ar, nb);
    s.w.bin_items = carve<int>(ar, kk);
    s.w.sorted = carve<double>(ar, kk * 5);
    if (from_bgr) s.lab = carve<uint8_t>(ar, (size_t)rows * cols * 3 * n);
    return s;
}

// Slic::generate_superpixels of n frames (arguments checked, 1 <= n <= 65535, at most the frames `s` was carved for) into
// `labels` (and `centers` when given): on the Lab frames `img` (dense), or, with from_bgr, on the cvtColor(COLOR_BGR2Lab)
// of the BGR frames `img` (pitch and frame stride in bytes), made into `s.lab` first
int enqueue_slic(const SlicBuffers& s, const uint8_t* img, size_t pitch, size_t fstride, bool from_bgr, int rows, int cols, int n, int step,
                 int nc, int iterations, int32_t* labels, double* centers, cudaStream_t st) {
    const int k = dcmt::slic_center_count(rows, cols, step);
    if (from_bgr) {
        const size_t lab_pitch = (size_t)cols * 3;
        API_CUDA(dcmt::color_bgr2lab(img, pitch, fstride, s.lab, lab_pitch, lab_pitch * rows, rows, cols, n, st), "BGR2Lab launch");
    }
    API_CUDA(dcmt::slic_run(from_bgr ? s.lab : img, rows, cols, n, step, nc, iterations, labels, k, s.w, st), "SLIC launch");
    if (centers && k > 0)
        API_CUDA(cudaMemcpyAsync(centers, s.w.centers, (size_t)k * n * 5 * sizeof(double), cudaMemcpyDeviceToDevice, st), "centre copy");
    return DCMT_OK;
}

// ---- the batched LiDAR projection, checked and enqueued on an arena its caller holds (dcmt_lidar_project_batch_f32 and the
// stereo chain).  max_clouds: 65535 for one launch; the chain runs in chunks and has no limit.
int check_project_batch(const float* points, int max_points, size_t cloud_stride_points, int n_clouds, int max_clouds, const float* T_host,
                        const float* P_host, int rows, int cols) {
    if ((!points && max_points > 0) || !T_host || !P_host) return fail(DCMT_E_BADARG, "null pointer");
    if (max_points < 0 || n_clouds < 0) return fail(DCMT_E_BADARG, "max_points %d, n_clouds %d", max_points, n_clouds);
    if (n_clouds > max_clouds) return fail(DCMT_E_UNSUPPORTED, "at most %d clouds per call", max_clouds);
    if (n_clouds > 1 && cloud_stride_points < (size_t)max_points) return fail(DCMT_E_BADARG, "cloud_stride_points %zu < max_points %d", cloud_stride_points, max_points);
    int rc = check_planes(rows, cols, 1);
    if (rc) return rc;
    if ((size_t)rows * (size_t)cols > (size_t)1 << 30) return fail(DCMT_E_UNSUPPORTED, "frame larger than 2^30 pixels");
    return DCMT_OK;
}

// the keys and min / max words of up to n clouds
dcmt::ProjectWork carve_project(Arena* ar, int rows, int cols, int n) {
    return dcmt::ProjectWork{carve<unsigned long long>(ar, dcmt::project_key_count(rows, cols) * n), carve<unsigned>(ar, 8 * (size_t)n)};
}

// the projection of n (1..65535, at most what `w` was carved for) clouds on checked arguments and 16-byte aligned points
int enqueue_project_batch(const dcmt::ProjectWork& w, const float* points, const int32_t* counts_dev, int max_points, size_t cloud_stride_points,
                          int n, const float* T_host, const float* P_host, int rows, int cols, float* projected, float* normalized, float norm_a,
                          float norm_b, int32_t* n_projected, cudaStream_t st) {
    return cuda_rc(dcmt::project_run_batch(points, max_points, counts_dev, cloud_stride_points, n, T_host, P_host, rows, cols, projected,
                                           normalized, norm_a, norm_b, n_projected, w, st),
                   "projection launch");
}

// device-pointer driver of the dcmt_interpolate_with_superpixels_bgr_* entry points (uint16 input: never synchronises).
// Chunks of the completion's size, each in one workspace of the caller's stream: Lab frames, labels, SLIC's work arrays
// and the completion workspace; BGR2Lab, SLIC and the guided completion run on that stream.
int run_completion_bgr(CompletionCall cc, InDesc in, OutDesc out, int n_frames, int32_t* stats, cudaStream_t st) {
    int rc = validate_completion(cc, &in, &out, n_frames);
    if (rc) return rc;
    if (n_frames == 0) return DCMT_OK;
    if ((rc = check_device())) return rc;
    API_CUDA(dcmt::generic_configure(), "kernel attribute setup");
    API_CUDA(dcmt::q8_configure(), "kernel attribute setup");
    cc.flags = input_path(in, cc.flags);
    const BgrFront& fr = *cc.front;
    const size_t fpix = (size_t)cc.rows * cc.cols;
    const int chunk = chunk_frames(cc.rows, cc.cols, n_frames, fused_applies(cc));
    for (int f0 = 0; f0 < n_frames; f0 += chunk) {
        const int nf = std::min(chunk, n_frames - f0);
        int32_t* labels = nullptr;
        SlicBuffers s;
        CompletionWork w;
        if ((rc = acquire_carved(st, [&](Arena* a) {  // stream order: the previous chunk is done with the arena
                 if (cc.guided) {
                     labels = carve<int32_t>(a, fpix * chunk);
                     s = carve_slic(a, cc.rows, cc.cols, chunk, fr.step, true);
                 }
                 w = carve_completion(a, cc, chunk, in.u, out.u);
             })))
            return rc;
        if (cc.guided && (rc = enqueue_slic(s, fr.bgr + (size_t)f0 * fr.fstride, fr.pitch, fr.fstride, true, cc.rows, cc.cols, nf, fr.step,
                                            fr.nc, fr.iterations, labels, nullptr, st)))
            return rc;
        if ((rc = enqueue_completion(cc, w, in.frames_from((size_t)f0), labels, out.frames_from((size_t)f0), nf,
                                     stats ? stats + (size_t)f0 * DCMT_STATS_STRIDE : nullptr, nullptr, nullptr, nullptr, st)))
            return rc;
    }
    return DCMT_OK;
}

// ---- host-pointer driver: chunks of frames flow H2D -> kernels -> D2H round-robin over three internal
// streams per device, so the copies of one chunk overlap the kernels of another.  Copies are asynchronous when the
// caller's buffers are page-locked (e.g. torch pinned memory); pageable buffers work, just slower.
//
// The same driver serves one device (the *_host entry points: the current device) and several (the *_host_multi entry
// points): the frames of the call are split into one contiguous block per device and the chunks of the blocks are
// enqueued round-robin by the calling thread -- every copy and launch is asynchronous, so one thread keeps all
// devices busy; there is no exchange between devices (frames are independent).
//
// Thread safety: the internal streams, their arenas and the pinned flag buffer are per device, so the host-pointer
// entry points take a per-device mutex for the duration of the call (several devices: in ascending device order).
// Two threads driving two different devices run concurrently; two threads on the same device take turns.
constexpr int kHostStreams = 3;
struct HostStreams {
    cudaStream_t s[kHostStreams];
};
std::map<int, HostStreams> g_host_streams;
std::map<int, std::mutex> g_host_mu;  // guarded by g_mu for insertion; std::map never moves its nodes

int host_streams(HostStreams** out) {
    int dev = 0;
    API_CUDA(cudaGetDevice(&dev), "cudaGetDevice");
    std::lock_guard<std::mutex> lk(g_mu);
    auto it = g_host_streams.find(dev);
    if (it == g_host_streams.end()) {
        HostStreams hs{};
        for (int i = 0; i < kHostStreams; ++i) API_CUDA(cudaStreamCreateWithFlags(&hs.s[i], cudaStreamNonBlocking), "cudaStreamCreate");
        it = g_host_streams.emplace(dev, hs).first;
    }
    *out = &it->second;
    return DCMT_OK;
}

int host_chunk_frames(int rows, int cols, int n_frames) {
    // pixels per chunk of the host pipeline (DCMT_HOST_CHUNK_MPX to override): small enough that filling and draining
    // the three-stage pipeline costs little, large enough for full-rate DMA and a few waves of CTAs
    static const long env = [] {
        const char* s = getenv("DCMT_HOST_CHUNK_MPX");
        return s ? atol(s) : 0L;
    }();
    const size_t px = env > 0 ? (size_t)env << 20 : (size_t)16 << 20;
    long c = (long)(px / ((size_t)rows * cols) + 1);
    if (c > n_frames) c = n_frames;
    if (c > 65535) c = 65535;
    return (int)(c < 1 ? 1 : c);
}

// One device of a host-pointer call.
struct Lane {
    int dev = 0;
    HostStreams* hs = nullptr;
    int f_begin = 0, f_end = 0;  // frames of the call served by this device
    int next = 0, slot = 0;      // next frame to enqueue, stream slot of the next chunk
    int32_t* h_flags = nullptr;  // pinned, one per frame of the lane (fused AUTO path)
};

// Scope of a host-pointer call: resolves the device list, takes the per-device mutexes, and on the way out -- success
// or error -- drains every internal stream of every device it touched (so no copy into the caller's buffers is still
// in flight after the function has returned) and restores the caller's current device.
class HostCall {
   public:
    ~HostCall() {
        drain();
        if (restore_ >= 0) cudaSetDevice(restore_);
        for (auto it = locks_.rbegin(); it != locks_.rend(); ++it) (*it)->unlock();
    }
    // devices == nullptr: n_devices <= 0 -> the current device; otherwise the first n_devices visible devices
    int open(const int* devices, int n_devices, bool all_if_null) {
        int rc = check_device();
        if (rc) return rc;
        int count = 0, cur = 0;
        API_CUDA(cudaGetDeviceCount(&count), "cudaGetDeviceCount");
        API_CUDA(cudaGetDevice(&cur), "cudaGetDevice");
        restore_ = cur;
        std::vector<int> ids;
        if (devices) {
            if (n_devices < 1) return fail(DCMT_E_BADARG, "n_devices must be >= 1 with an explicit device list (got %d)", n_devices);
            ids.assign(devices, devices + n_devices);
        } else if (all_if_null) {
            const int n = n_devices > 0 ? n_devices : count;
            if (n > count) return fail(DCMT_E_BADARG, "%d devices requested, %d visible", n, count);
            for (int d = 0; d < n; ++d) ids.push_back(d);
        } else {
            ids.push_back(cur);
        }
        std::vector<int> sorted = ids;
        std::sort(sorted.begin(), sorted.end());
        for (size_t i = 0; i < sorted.size(); ++i) {
            if (sorted[i] < 0 || sorted[i] >= count) return fail(DCMT_E_BADARG, "device %d out of range (%d visible)", sorted[i], count);
            if (i && sorted[i] == sorted[i - 1]) return fail(DCMT_E_BADARG, "device %d listed twice", sorted[i]);
        }
        for (int d : sorted) {  // ascending order: two calls with overlapping device sets cannot deadlock
            std::mutex* m;
            {
                std::lock_guard<std::mutex> lk(g_mu);
                m = &g_host_mu[d];
            }
            m->lock();
            locks_.push_back(m);
        }
        lanes.resize(ids.size());
        for (size_t i = 0; i < ids.size(); ++i) {
            lanes[i].dev = ids[i];
            API_CUDA(cudaSetDevice(ids[i]), "cudaSetDevice");
            if ((rc = host_streams(&lanes[i].hs))) return rc;
        }
        return DCMT_OK;
    }
    // contiguous blocks of frames, sizes differing by at most one
    void split(int n_frames) {
        const int n = (int)lanes.size();
        for (int i = 0; i < n; ++i) {
            lanes[i].f_begin = (int)((long long)n_frames * i / n);
            lanes[i].f_end = (int)((long long)n_frames * (i + 1) / n);
            lanes[i].next = lanes[i].f_begin;
        }
    }
    int use(Lane& l) {
        API_CUDA(cudaSetDevice(l.dev), "cudaSetDevice");
        drained_ = false;  // the caller is about to enqueue on this lane
        return DCMT_OK;
    }
    // waits for all enqueued work; the first error wins
    int finish() {
        cudaError_t first = cudaSuccess;
        for (Lane& l : lanes) {
            if (!l.hs) continue;
            cudaSetDevice(l.dev);
            for (int i = 0; i < kHostStreams; ++i) {
                const cudaError_t e = cudaStreamSynchronize(l.hs->s[i]);
                if (e != cudaSuccess && first == cudaSuccess) first = e;
            }
        }
        drained_ = true;
        return first == cudaSuccess ? DCMT_OK : cuda_fail(first, "kernel execution");
    }
    std::vector<Lane> lanes;

   private:
    void drain() {
        if (drained_) return;
        for (Lane& l : lanes) {
            if (!l.hs) continue;
            cudaSetDevice(l.dev);
            for (int i = 0; i < kHostStreams; ++i) cudaStreamSynchronize(l.hs->s[i]);
        }
        drained_ = true;
    }
    std::vector<std::mutex*> locks_;
    int restore_ = -1;
    bool drained_ = false;
};

int copy_frames_h2d(void* d, size_t d_pitch_bytes, const void* h, size_t h_pitch_bytes, size_t h_fstride_bytes, size_t row_bytes, int rows,
                    int nf, cudaStream_t st) {
    if (d_pitch_bytes == row_bytes && h_pitch_bytes == row_bytes && h_fstride_bytes == row_bytes * rows) {
        API_CUDA(cudaMemcpyAsync(d, h, row_bytes * rows * nf, cudaMemcpyHostToDevice, st), "host to device copy");
    } else if (h_fstride_bytes == h_pitch_bytes * (size_t)rows) {  // frames back to back: one 2-D copy for the whole chunk
        API_CUDA(cudaMemcpy2DAsync(d, d_pitch_bytes, h, h_pitch_bytes, row_bytes, (size_t)rows * nf, cudaMemcpyHostToDevice, st),
                 "host to device copy");
    } else {
        for (int f = 0; f < nf; ++f)
            API_CUDA(cudaMemcpy2DAsync(static_cast<char*>(d) + (size_t)f * rows * d_pitch_bytes, d_pitch_bytes,
                                       static_cast<const char*>(h) + (size_t)f * h_fstride_bytes, h_pitch_bytes, row_bytes, rows,
                                       cudaMemcpyHostToDevice, st),
                     "host to device copy");
    }
    return DCMT_OK;
}

// device frames are back to back with rows of d_pitch_bytes
int copy_frames_d2h(void* h, size_t h_pitch_bytes, size_t h_fstride_bytes, const void* d, size_t d_pitch_bytes, size_t row_bytes, int rows,
                    int nf, cudaStream_t st) {
    if (d_pitch_bytes == row_bytes && h_pitch_bytes == row_bytes && h_fstride_bytes == row_bytes * rows) {
        API_CUDA(cudaMemcpyAsync(h, d, row_bytes * rows * nf, cudaMemcpyDeviceToHost, st), "device to host copy");
    } else if (h_fstride_bytes == h_pitch_bytes * (size_t)rows) {
        API_CUDA(cudaMemcpy2DAsync(h, h_pitch_bytes, d, d_pitch_bytes, row_bytes, (size_t)rows * nf, cudaMemcpyDeviceToHost, st), "device to host copy");
    } else {
        for (int f = 0; f < nf; ++f)
            API_CUDA(cudaMemcpy2DAsync(static_cast<char*>(h) + (size_t)f * h_fstride_bytes, h_pitch_bytes,
                                       static_cast<const char*>(d) + (size_t)f * rows * d_pitch_bytes, d_pitch_bytes, row_bytes, rows,
                                       cudaMemcpyDeviceToHost, st),
                     "device to host copy");
    }
    return DCMT_OK;
}

// One caller buffer of a single-shot host call: `rows` rows of `row_bytes`, `pitch` bytes apart on the host, packed on the
// device.
struct Staged {
    const void* from;     // copied to the device before the work (nullptr: not read)
    void* to;             // copied back after the work (nullptr: not written back)
    size_t pitch, row_bytes, rows;
    void* dev = nullptr;  // set by run_staged
};

// Driver of the single-shot host entry points, called on validated arguments: a HostCall on the current device, the staging
// of `bufs` carved from the arena of the lane's second stream, then H2D, work(stream) and D2H on the first stream, whose
// arena is left to the work's own workspace; HostCall::finish waits for all of it.
template <class Work>
int run_staged(std::initializer_list<Staged*> bufs, Work&& work) {
    HostCall call;
    int rc = call.open(nullptr, 0, false);
    if (rc) return rc;
    Lane& l = call.lanes[0];
    const cudaStream_t st = l.hs->s[0];
    if ((rc = acquire_carved(l.hs->s[1], [&](Arena* a) {
             for (Staged* b : bufs) b->dev = carve<char>(a, b->rows * b->row_bytes);
         })) ||
        (rc = call.use(l)))
        return rc;
    // one copy when the host rows are packed, a 2-D copy otherwise
    auto copy = [st](void* dst, size_t dst_pitch, const void* src, size_t src_pitch, const Staged* b, cudaMemcpyKind kind) {
        return dst_pitch == src_pitch ? cudaMemcpyAsync(dst, src, b->rows * b->row_bytes, kind, st)
                                      : cudaMemcpy2DAsync(dst, dst_pitch, src, src_pitch, b->row_bytes, b->rows, kind, st);
    };
    for (const Staged* b : bufs)
        if (b->from) API_CUDA(copy(b->dev, b->row_bytes, b->from, b->pitch, b, cudaMemcpyHostToDevice), "host to device copy");
    if ((rc = work(st))) return rc;
    for (const Staged* b : bufs)
        if (b->to) API_CUDA(copy(b->to, b->pitch, b->dev, b->row_bytes, b, cudaMemcpyDeviceToHost), "device to host copy");
    return call.finish();
}

// The host chunk pipeline of a host-pointer call of n_frames frames: opens the call (devices, n_devices and multi as
// HostCall::open takes them), gives every device a contiguous block of the frames and enqueues host chunks
// (host_chunk_frames of the longest block) round-robin over the devices, each device's chunks on its three streams in
// turn.  chunk(lane, stream, f0, nf, frames, level) enqueues frames [f0, f0 + nf) at path `level` in a workspace sized for
// `frames` frames.  configure: the completion kernels' attributes are set on every device first.  flagged: every lane
// gets a pinned flag buffer (Lane::h_flags) that the chunks of a pass fill with the frames they did not serve; after the
// pass those frames are redone one level down (path_below), in runs of consecutive frames cut into host chunks, on the
// device that served them, until a level leaves none.
template <class Chunk>
int run_host_chunks(int n_frames, int rows, int cols, const int* devices, int n_devices, bool multi, bool configure, bool flagged, int level,
                    Chunk&& chunk) {
    HostCall call;
    int rc = call.open(devices, n_devices, multi);
    if (rc) return rc;
    call.split(n_frames);
    int longest = 0;
    for (Lane& l : call.lanes) longest = std::max(longest, l.f_end - l.f_begin);
    const int hc = host_chunk_frames(rows, cols, longest);
    for (Lane& l : call.lanes) {
        if (l.f_end == l.f_begin) continue;
        if ((rc = call.use(l))) return rc;
        if (configure) {
            API_CUDA(dcmt::generic_configure(), "kernel attribute setup");
            API_CUDA(dcmt::q8_configure(), "kernel attribute setup");
        }
        if (flagged && (rc = pinned_flags(nullptr, (size_t)(l.f_end - l.f_begin), &l.h_flags))) return rc;
    }
    // on the lane's next stream: stream order protects the reuse of its arena by the chunk three steps later
    auto enqueue = [&](Lane& l, int f0, int nf, int frames, int lv) {
        if (int rc2 = call.use(l)) return rc2;
        const cudaStream_t st = l.hs->s[l.slot];
        l.slot = (l.slot + 1) % kHostStreams;
        return chunk(l, st, f0, nf, frames, lv);
    };
    for (bool more = true; more;) {
        more = false;
        for (Lane& l : call.lanes) {
            if (l.next >= l.f_end) continue;
            more = true;
            const int f0 = l.next, nf = std::min(hc, l.f_end - f0);
            l.next += nf;
            if ((rc = enqueue(l, f0, nf, hc, level))) return rc;
        }
    }
    if ((rc = call.finish())) return rc;
    for (int lv = path_below(level); flagged && lv >= 0; lv = path_below(lv)) {
        // the runs are fixed before anything is enqueued: a pass may write the flags it reads
        std::vector<std::pair<Lane*, Run>> runs;
        for (Lane& l : call.lanes)
            for (const Run& r : flagged_runs(l.h_flags, l.f_end - l.f_begin)) runs.push_back({&l, Run{l.f_begin + r.f, l.f_begin + r.e}});
        if (runs.empty()) break;
        for (const auto& [l, r] : runs) {
            const int rhc = host_chunk_frames(rows, cols, r.e - r.f);
            for (int f = r.f; f < r.e; f += rhc)
                if ((rc = enqueue(*l, f, std::min(rhc, r.e - f), rhc, lv))) return rc;
        }
        if ((rc = call.finish())) return rc;
    }
    return DCMT_OK;
}

// Host-pointer driver of every completion entry point.  Device staging rows are packed for float32 input and padded to
// 16 bytes for uint16 input (vector loads in k_q8_front).
// copy_only: the same buffers, chunking and streams with the kernels left out -- the ceiling the host <-> device links put
// on the end-to-end rate (dcmt_debug_host_copy_*).  An output of the input's type echoes the input; a float32 output of
// uint16 input is zeroed.
int run_completion_host(CompletionCall cc, InDesc in, OutDesc out, int n_frames, int32_t* stats, const int* devices = nullptr,
                        int n_devices = 0, bool multi = false, bool copy_only = false) {
    int rc = validate_completion(cc, &in, &out, n_frames);
    if (rc) return rc;
    if (n_frames == 0) return DCMT_OK;
    const int rows = cc.rows, cols = cc.cols;
    const size_t fpix = (size_t)rows * cols;
    const size_t in_elem = in.elem(), out_elem = out.elem();
    const size_t d_pitch = in.u ? pad8(cols) : (size_t)cols;  // elements of a device staging row of the input
    cc.flags = input_path(in, cc.flags);
    const bool flagged = writes_flags(cc, in.f, copy_only);
    // labels made from BGR frames on the device (staged packed, 3 bytes per pixel) instead of copied in
    const BgrFront* front = cc.guided ? cc.front : nullptr;
    const size_t bgr_row = (size_t)cols * 3;
    // H2D, kernels, D2H; the arena holds the staging of input, output, labels, stats, flags and BGR frames, then the workspace
    auto chunk = [&](Lane& l, cudaStream_t st, int f0, int nf, int hc, int level) -> int {
        CompletionCall c2 = cc;
        c2.flags = level;
        const bool flags2 = writes_flags(c2, in.f, copy_only);  // the generic redo pass reports no flags
        char *d_in, *d_out;
        int32_t *d_lab, *d_stats, *d_flags;
        uint8_t* d_bgr;
        SlicBuffers s{};
        CompletionWork w{};
        int rc2 = acquire_carved(st, [&](Arena* a) {
            d_in = carve<char>(a, (size_t)rows * d_pitch * hc * in_elem);
            d_out = carve<char>(a, fpix * hc * out_elem);
            d_lab = cc.guided ? carve<int32_t>(a, fpix * hc) : nullptr;
            d_stats = carve<int32_t>(a, (size_t)hc * DCMT_STATS_STRIDE);
            d_flags = flagged ? carve<int32_t>(a, (size_t)hc) : nullptr;
            d_bgr = front ? carve<uint8_t>(a, bgr_row * rows * hc) : nullptr;
            if (front) s = carve_slic(a, rows, cols, hc, front->step, true);
            if (!copy_only) w = carve_completion(a, c2, hc, in.u, out.u);
        });
        if (rc2) return rc2;
        if (front && (rc2 = copy_frames_h2d(d_bgr, bgr_row, front->bgr + (size_t)f0 * front->fstride, front->pitch, front->fstride, bgr_row,
                                            rows, nf, st)))
            return rc2;
        const InDesc hi = in.frames_from((size_t)f0);
        if ((rc2 = copy_frames_h2d(d_in, d_pitch * in_elem, hi.ptr(), in.pitch * in_elem, in.fstride * in_elem, cols * in_elem, rows, nf, st)))
            return rc2;
        if (front) {
            if ((rc2 = enqueue_slic(s, d_bgr, bgr_row, bgr_row * rows, true, rows, cols, nf, front->step, front->nc, front->iterations, d_lab,
                                    nullptr, st)))
                return rc2;
        } else if (cc.guided) {
            API_CUDA(cudaMemcpyAsync(d_lab, cc.labels + (size_t)f0 * fpix, fpix * nf * sizeof(int32_t), cudaMemcpyHostToDevice, st),
                     "host to device copy");
        }
        size_t d_out_pitch = cols;  // elements
        if (copy_only && in_elem == out_elem) {
            d_out = d_in;
            d_out_pitch = d_pitch;
        } else if (copy_only) {
            API_CUDA(cudaMemsetAsync(d_out, 0, fpix * nf * out_elem, st), "memset");
        } else {
            const InDesc di = in.u ? InDesc{nullptr, reinterpret_cast<uint16_t*>(d_in), d_pitch, rows * d_pitch}
                                   : InDesc{reinterpret_cast<float*>(d_in), nullptr, d_pitch, rows * d_pitch};
            const OutDesc dout = out.u ? OutDesc{nullptr, reinterpret_cast<uint16_t*>(d_out), (size_t)cols, fpix}
                                       : OutDesc{reinterpret_cast<float*>(d_out), nullptr, (size_t)cols, fpix};
            if ((rc2 = enqueue_completion(c2, w, di, d_lab, dout, nf, stats ? d_stats : nullptr, flags2 ? d_flags : nullptr, nullptr, nullptr, st)))
                return rc2;
        }
        if (flags2)
            API_CUDA(cudaMemcpyAsync(l.h_flags + (f0 - l.f_begin), d_flags, (size_t)nf * sizeof(int32_t), cudaMemcpyDeviceToHost, st),
                     "flag readback");
        const OutDesc ho = out.frames_from((size_t)f0);
        if ((rc2 = copy_frames_d2h(ho.ptr(), out.pitch * out_elem, out.fstride * out_elem, d_out, d_out_pitch * out_elem, cols * out_elem,
                                   rows, nf, st)))
            return rc2;
        if (stats && !copy_only)
            API_CUDA(cudaMemcpyAsync(stats + (size_t)f0 * DCMT_STATS_STRIDE, d_stats, (size_t)nf * DCMT_STATS_STRIDE * sizeof(int32_t),
                                     cudaMemcpyDeviceToHost, st),
                     "device to host copy");
        return DCMT_OK;
    };
    return run_host_chunks(n_frames, rows, cols, devices, n_devices, multi, true, flagged, cc.flags, chunk);
}

// ---- the stereo program's per-frame chain (dcmt_stereo_chain_f32*, main_sl.cpp:435-563 + :1162-1253): batched projection
// + cv::normalize, SLIC of the left frame from BGR, the guided completion of the normalised floats, BGR2GRAY of both frames
// and the stereo refinement, with every intermediate in the workspace.
struct StereoChain {
    const float* points;
    const int32_t* counts;  // n_points per cloud (device array on the device form, host array on the host forms) or null
    int max_points;
    size_t cloud_stride;  // points
    const float *T, *P;
    float norm_a, norm_b;
    const uint8_t *left, *right;
    size_t bgr_pitch, bgr_fstride;  // bytes; the ABI's 0 = dense until validate_stereo_chain fills them in
    float *depth, *disp;
    int rows, cols, n_frames, step, nc, iterations, use_superpixel, flags;
    const dcmt_stereo_params* prm;
    int32_t* stats;
};

// Checks a chain call: the projection's arguments, the other pointers, flags, the refinement's parameters, SLIC's limits,
// BGR2GRAY's rows, the BGR geometry and overlap of the outputs, in this order; on the host forms (host_counts) the cloud
// sizes last, the only caller data a check reads.
int validate_stereo_chain(StereoChain& c, bool host_counts) {
    int rc = check_project_batch(c.points, c.max_points, c.cloud_stride, c.n_frames, INT32_MAX, c.T, c.P, c.rows, c.cols);
    if (rc) return rc;
    if (!c.left || !c.right || !c.depth || !c.prm) return fail(DCMT_E_BADARG, "null pointer");
    if (c.flags < DCMT_PATH_AUTO || c.flags > DCMT_PATH_RANK) return fail(DCMT_E_BADARG, "flags %d", c.flags);
    if (c.flags == DCMT_PATH_FUSED) return fail(DCMT_E_BADARG, "DCMT_PATH_FUSED: the normalised projection is not strict q8");
    if (c.prm->num_iterations < 0) return fail(DCMT_E_BADARG, "num_iterations %d", c.prm->num_iterations);
    if ((rc = check_slic(c.rows, c.cols, c.step, c.nc, c.iterations))) return rc;
    if (c.rows > 65535) return fail(DCMT_E_UNSUPPORTED, "at most 65535 rows");
    size_t bgr_span = 0;
    if ((rc = check_bgr_geometry(c.rows, c.cols, &c.bgr_pitch, &c.bgr_fstride, c.n_frames, &bgr_span))) return rc;
    if (c.n_frames) {
        const size_t plane = (size_t)c.rows * c.cols * c.n_frames * sizeof(float);
        const size_t cloud_span = c.points ? ((size_t)(c.n_frames - 1) * c.cloud_stride + c.max_points) * 16 : 0;
        const size_t count_span = c.counts ? (size_t)c.n_frames * sizeof(int32_t) : 0;
        for (const float* o : {c.depth, c.disp}) {
            if (!o) continue;
            if (overlaps(o, plane, c.points, cloud_span) || overlaps(o, plane, c.counts, count_span) || overlaps(o, plane, c.left, bgr_span) ||
                overlaps(o, plane, c.right, bgr_span))
                return fail(DCMT_E_BADARG, "an output overlaps an input");
        }
        if (c.disp && overlaps(c.depth, plane, c.disp, plane)) return fail(DCMT_E_BADARG, "depth_out and disp_out overlap");
    }
    if (host_counts && c.counts)
        for (int f = 0; f < c.n_frames; ++f)
            if (c.counts[f] < 0 || c.counts[f] > c.max_points)
                return fail(DCMT_E_BADARG, "n_points[%d] = %d outside [0, max_points %d]", f, c.counts[f], c.max_points);
    return DCMT_OK;
}

// The completion of the chain: the guided call on the normalised floats, AUTO going straight to the dictionary level (the
// strict-q8 pass would fail on every frame with points; every level gives the same bits)
CompletionCall chain_completion(const StereoChain& c) {
    return CompletionCall{nullptr, dcmt::slic_center_count(c.rows, c.cols, c.step), c.use_superpixel != 0, c.rows, c.cols, DCMT_BLUR_GAUSSIAN,
                          c.flags == DCMT_PATH_GENERIC ? DCMT_PATH_GENERIC : DCMT_PATH_RANK};
}

// Device pointers of nf frames of the chain: 16-byte aligned clouds `cloud_stride` points apart (counts: device array or
// null), the BGR pairs, and dense outputs (disp, stats and the completion's "not served" flags optional)
struct ChainFrames {
    const float* points;
    const int32_t* counts;
    size_t cloud_stride;
    const uint8_t *left, *right;
    size_t bgr_pitch, bgr_fstride;
    float *depth, *disp;
    int32_t *stats, *flags;
};

// The intermediates of chunks of up to `chunk` frames: normalised plane, completed depth, the two gray planes, the
// projection's keys and min / max words, labels, Lab frames and SLIC's work arrays (guided only), and the completion's
// workspace.  About 37 bytes per pixel, 4.8 GB at 313 KITTI frames.
struct ChainWork {
    float *nrm, *dense;
    uint8_t *gray_l, *gray_r;
    dcmt::ProjectWork proj;
    int32_t* labels;
    SlicBuffers slic;
    CompletionWork completion;
};

ChainWork carve_chain(Arena* ar, const StereoChain& c, const CompletionCall& cc, int chunk) {
    const size_t px = (size_t)c.rows * c.cols * chunk;
    return ChainWork{carve<float>(ar, px), carve<float>(ar, px), carve<uint8_t>(ar, px), carve<uint8_t>(ar, px), carve_project(ar, c.rows, c.cols, chunk),
                     cc.guided ? carve<int32_t>(ar, px) : nullptr, cc.guided ? carve_slic(ar, c.rows, c.cols, chunk, c.step, true) : SlicBuffers{},
                     carve_completion(ar, cc, chunk, false, false)};
}

// one chunk (1 <= nf <= 65535 frames, at most what `w` was carved for) of the chain on one stream
int enqueue_chain(const StereoChain& c, const CompletionCall& cc, const ChainWork& w, const ChainFrames& io, int nf, cudaStream_t st) {
    const int rows = c.rows, cols = c.cols;
    const size_t fpix = (size_t)rows * cols;
    int rc = enqueue_project_batch(w.proj, io.points, io.counts, c.max_points, io.cloud_stride, nf, c.T, c.P, rows, cols, nullptr, w.nrm, c.norm_a,
                                   c.norm_b, nullptr, st);
    if (rc) return rc;
    if (cc.guided &&
        (rc = enqueue_slic(w.slic, io.left, io.bgr_pitch, io.bgr_fstride, true, rows, cols, nf, c.step, c.nc, c.iterations, w.labels, nullptr, st)))
        return rc;
    if ((rc = enqueue_completion(cc, w.completion, InDesc{w.nrm, nullptr, (size_t)cols, fpix}, w.labels, OutDesc{w.dense, nullptr, (size_t)cols, fpix},
                                 nf, io.stats, io.flags, nullptr, nullptr, st)))
        return rc;
    API_CUDA(dcmt::stereo_bgr2gray(io.left, io.bgr_pitch, io.bgr_fstride, w.gray_l, cols, fpix, rows, cols, nf, st), "BGR2GRAY launch");
    API_CUDA(dcmt::stereo_bgr2gray(io.right, io.bgr_pitch, io.bgr_fstride, w.gray_r, cols, fpix, rows, cols, nf, st), "BGR2GRAY launch");
    const dcmt_stereo_params& p = *c.prm;
    API_CUDA(dcmt::stereo_refine(w.dense, w.gray_l, w.gray_r, io.depth, io.disp, rows, cols, nf, p.baseline, p.focal, p.damp_factor, p.err_clip,
                                 p.depth_clip, p.num_iterations, p.final_gauss, st),
             "stereo refine launch");
    return DCMT_OK;
}

// Device-pointer driver of dcmt_stereo_chain_f32: chunks of the generic pipeline's size (chunk_frames) on the caller's
// stream.  On the dictionary path the "not served" flags of the whole call sit at the start of every chunk's arena (the
// same bytes each time: every chunk carves the same workspace) and are read back once; those frames are redone through
// the chain one level down, on the generic pipeline, which reports no flags.
int run_stereo_chain(StereoChain c, cudaStream_t st) {
    int rc = validate_stereo_chain(c, false);
    if (rc) return rc;
    if (c.points && (reinterpret_cast<uintptr_t>(c.points) & 15)) return fail(DCMT_E_BADARG, "points must be 16-byte aligned");
    if (c.n_frames == 0) return DCMT_OK;
    if ((rc = check_device())) return rc;
    API_CUDA(dcmt::generic_configure(), "kernel attribute setup");
    API_CUDA(dcmt::q8_configure(), "kernel attribute setup");
    CompletionCall cc = chain_completion(c);
    const int n = c.n_frames, chunk = chunk_frames(c.rows, c.cols, n, false);
    const bool flagged = writes_flags(cc, true, false);
    const size_t fpix = (size_t)c.rows * c.cols;
    auto frames = [&](int f0, int32_t* flags) {
        return ChainFrames{c.points ? c.points + (size_t)f0 * c.cloud_stride * 4 : nullptr, c.counts ? c.counts + f0 : nullptr, c.cloud_stride,
                           c.left + (size_t)f0 * c.bgr_fstride, c.right + (size_t)f0 * c.bgr_fstride, c.bgr_pitch, c.bgr_fstride,
                           c.depth + (size_t)f0 * fpix, c.disp ? c.disp + (size_t)f0 * fpix : nullptr,
                           c.stats ? c.stats + (size_t)f0 * DCMT_STATS_STRIDE : nullptr, flags};
    };
    int32_t* d_flags = nullptr;
    ChainWork w;
    for (int f0 = 0; f0 < n; f0 += chunk) {
        if ((rc = acquire_carved(st, [&](Arena* a) {  // stream order: the previous chunk is done with the arena
                 d_flags = flagged ? carve<int32_t>(a, (size_t)n) : nullptr;
                 w = carve_chain(a, c, cc, chunk);
             })))
            return rc;
        if ((rc = enqueue_chain(c, cc, w, frames(f0, d_flags ? d_flags + f0 : nullptr), std::min(chunk, n - f0), st))) return rc;
    }
    if (!flagged) return DCMT_OK;
    int32_t* h_flags = nullptr;
    if ((rc = pinned_flags(st, (size_t)n, &h_flags))) return rc;
    API_CUDA(cudaMemcpyAsync(h_flags, d_flags, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, st), "flag readback");
    API_CUDA(cudaStreamSynchronize(st), "kernel execution");
    cc.flags = path_below(cc.flags);
    for (const Run& r : flagged_runs(h_flags, n)) {
        for (int f0 = r.f; f0 < r.e; f0 += chunk) {
            if ((rc = acquire_carved(st, [&](Arena* a) { w = carve_chain(a, c, cc, chunk); }))) return rc;
            if ((rc = enqueue_chain(c, cc, w, frames(f0, nullptr), std::min(chunk, r.e - f0), st))) return rc;
        }
    }
    return DCMT_OK;
}

// Host-pointer driver of dcmt_stereo_chain_f32_host[_multi] on the host chunk pipeline.  A chunk stages n_points[c] * 16
// bytes of each cloud (max_points apart), the cloud sizes and both BGR frames (packed), runs the chain into its arena and
// copies depth, disparity, stats and the dictionary's flags back.
int run_stereo_chain_host(StereoChain c, const int* devices = nullptr, int n_devices = 0, bool multi = false) {
    int rc = validate_stereo_chain(c, true);
    if (rc) return rc;
    if (c.n_frames == 0) return DCMT_OK;
    if (c.n_frames == 1) c.cloud_stride = c.max_points;  // one cloud: the ABI lets its stride be anything; staged clouds are max_points apart
    const int rows = c.rows, cols = c.cols;
    const size_t fpix = (size_t)rows * cols, bgr_row = (size_t)cols * 3, cloud_bytes = (size_t)c.max_points * 16;
    const CompletionCall cc = chain_completion(c);
    auto chunk = [&](Lane& l, cudaStream_t st, int f0, int nf, int hc, int level) -> int {
        CompletionCall c2 = cc;
        c2.flags = level;
        const bool flags2 = writes_flags(c2, true, false);
        const size_t px = fpix * hc;
        float *d_pts, *d_depth, *d_disp;
        int32_t *d_counts, *d_stats, *d_flags;
        uint8_t *d_left, *d_right;
        ChainWork w;
        int rc2 = acquire_carved(st, [&](Arena* a) {
            d_pts = carve<float>(a, (size_t)c.max_points * 4 * hc);
            d_counts = c.counts ? carve<int32_t>(a, (size_t)hc) : nullptr;
            d_left = carve<uint8_t>(a, bgr_row * rows * hc);
            d_right = carve<uint8_t>(a, bgr_row * rows * hc);
            d_depth = carve<float>(a, px);
            d_disp = c.disp ? carve<float>(a, px) : nullptr;
            d_stats = carve<int32_t>(a, (size_t)hc * DCMT_STATS_STRIDE);
            d_flags = flags2 ? carve<int32_t>(a, (size_t)hc) : nullptr;
            w = carve_chain(a, c, c2, hc);
        });
        if (rc2) return rc2;
        const float* h_pts = c.points ? c.points + (size_t)f0 * c.cloud_stride * 4 : nullptr;
        if (c.counts) {
            API_CUDA(cudaMemcpyAsync(d_counts, c.counts + f0, (size_t)nf * sizeof(int32_t), cudaMemcpyHostToDevice, st), "host to device copy");
            for (int i = 0; i < nf; ++i)
                if (c.counts[f0 + i] > 0)
                    API_CUDA(cudaMemcpyAsync(d_pts + (size_t)i * c.max_points * 4, h_pts + (size_t)i * c.cloud_stride * 4, (size_t)c.counts[f0 + i] * 16,
                                             cudaMemcpyHostToDevice, st),
                             "host to device copy");
        } else if (cloud_bytes > 0 &&
                   (rc2 = copy_frames_h2d(d_pts, cloud_bytes, h_pts, c.cloud_stride * 16, c.cloud_stride * 16, cloud_bytes, 1, nf, st))) {
            return rc2;
        }
        if ((rc2 = copy_frames_h2d(d_left, bgr_row, c.left + (size_t)f0 * c.bgr_fstride, c.bgr_pitch, c.bgr_fstride, bgr_row, rows, nf, st)) ||
            (rc2 = copy_frames_h2d(d_right, bgr_row, c.right + (size_t)f0 * c.bgr_fstride, c.bgr_pitch, c.bgr_fstride, bgr_row, rows, nf, st)))
            return rc2;
        const ChainFrames io{d_pts, d_counts, (size_t)c.max_points, d_left, d_right, bgr_row, bgr_row * rows, d_depth, d_disp,
                             c.stats ? d_stats : nullptr, d_flags};
        if ((rc2 = enqueue_chain(c, c2, w, io, nf, st))) return rc2;
        if (flags2)
            API_CUDA(cudaMemcpyAsync(l.h_flags + (f0 - l.f_begin), d_flags, (size_t)nf * sizeof(int32_t), cudaMemcpyDeviceToHost, st), "flag readback");
        API_CUDA(cudaMemcpyAsync(c.depth + (size_t)f0 * fpix, d_depth, fpix * nf * sizeof(float), cudaMemcpyDeviceToHost, st), "device to host copy");
        if (c.disp)
            API_CUDA(cudaMemcpyAsync(c.disp + (size_t)f0 * fpix, d_disp, fpix * nf * sizeof(float), cudaMemcpyDeviceToHost, st), "device to host copy");
        if (c.stats)
            API_CUDA(cudaMemcpyAsync(c.stats + (size_t)f0 * DCMT_STATS_STRIDE, d_stats, (size_t)nf * DCMT_STATS_STRIDE * sizeof(int32_t),
                                     cudaMemcpyDeviceToHost, st),
                     "device to host copy");
        return DCMT_OK;
    };
    return run_host_chunks(c.n_frames, rows, cols, devices, n_devices, multi, true, writes_flags(cc, true, false), cc.flags, chunk);
}

// ---- evaluation: one device driver and one host driver behind every dcmt_evaluate_* entry point.  Each side is an InDesc:
// float32 metres or KITTI uint16 (metres * 256), with the ABI's pitch and frame stride in bytes (0 = dense) until
// validate_evaluation checks them against the side's element size and converts them to elements.  uint16 results come
// with a uint16 GT only (the entry points offer no other pair).
int validate_evaluation(InDesc* gt, InDesc* r, int rows, int cols, int n_frames, int mode, const void* results, size_t* gt_span,
                        size_t* r_span) {
    if (!gt->ptr() || !r->ptr() || !results) return fail(DCMT_E_BADARG, "null pointer");
    if (mode != DCMT_EVAL_GT_VALID && mode != DCMT_EVAL_BOTH_VALID) return fail(DCMT_E_BADARG, "mode %d", mode);
    Geometry g, q;
    int rc = check_geometry(rows, cols, gt->pitch, gt->fstride, n_frames, &g, gt->elem());
    if (rc) return rc;
    if ((rc = check_geometry(rows, cols, r->pitch, r->fstride, n_frames, &q, r->elem()))) return rc;
    gt->pitch = g.pitch;
    gt->fstride = g.fstride;
    r->pitch = q.pitch;
    r->fstride = q.fstride;
    *gt_span = g.span_bytes;
    *r_span = q.span_bytes;
    return DCMT_OK;
}

// One kind of evaluation: the size of its per-frame record and how its kernels are enqueued on validated arguments
// (n_frames >= 1): the reductions of dcmt_evaluate_* (EvalReductions) or the KITTI benchmark's figures (EvalKitti).
struct EvalKind {
    size_t rec_bytes;
    explicit EvalKind(size_t bytes) : rec_bytes(bytes) {}
    virtual int enqueue(const InDesc& gt, const InDesc& r, int rows, int cols, int n_frames, void* results, cudaStream_t st) const = 0;
};

// partial sums in the stream's arena, then the two kernels of evaluate.cu
struct EvalReductions : EvalKind {
    float tolerance;
    int mode;
    EvalReductions(float tol, int m) : EvalKind(sizeof(dcmt_eval_result)), tolerance(tol), mode(m) {}
    int enqueue(const InDesc& gt, const InDesc& r, int rows, int cols, int n_frames, void* results, cudaStream_t st) const override {
        double* partials = nullptr;
        if (int rc = acquire_carved(st, [&](Arena* a) { partials = carve<double>(a, dcmt::eval_partial_doubles(n_frames)); })) return rc;
        dcmt::EvalResult* out = static_cast<dcmt::EvalResult*>(results);
        cudaError_t e;
        if (!gt.u)
            e = dcmt::eval_run(gt.f, gt.pitch, gt.fstride, r.f, r.pitch, r.fstride, rows, cols, n_frames, tolerance, mode, partials, out, st);
        else if (!r.u)
            e = dcmt::eval_run(gt.u, gt.pitch, gt.fstride, r.f, r.pitch, r.fstride, rows, cols, n_frames, tolerance, mode, partials, out, st);
        else
            e = dcmt::eval_run(gt.u, gt.pitch, gt.fstride, r.u, r.pitch, r.fstride, rows, cols, n_frames, tolerance, mode, partials, out, st);
        API_CUDA(e, "evaluation launch");
        return DCMT_OK;
    }
};

// partial sums, the first / last valid prediction rows and (rows of more than 262 144 columns) the blocks' validity bits
// in the stream's arena, then the three kernels of evaluate.cu
struct EvalKitti : EvalKind {
    EvalKitti() : EvalKind(sizeof(dcmt_kitti_metrics)) {}
    int enqueue(const InDesc& gt, const InDesc& r, int rows, int cols, int n_frames, void* results, cudaStream_t st) const override {
        const size_t nd = dcmt::kitti_partial_doubles(n_frames), nw = dcmt::kitti_bits_words(rows, cols, n_frames);
        double* partials = nullptr;
        int32_t* first_last = nullptr;
        unsigned* bits = nullptr;
        if (int rc = acquire_carved(st, [&](Arena* a) {
                partials = carve<double>(a, nd);
                first_last = carve<int32_t>(a, 2 * (size_t)n_frames);
                bits = nw ? carve<unsigned>(a, nw) : nullptr;
            }))
            return rc;
        dcmt::KittiMetrics* out = static_cast<dcmt::KittiMetrics*>(results);
        cudaError_t e;
        if (!gt.u)
            e = dcmt::kitti_run(gt.f, gt.pitch, gt.fstride, r.f, r.pitch, r.fstride, rows, cols, n_frames, partials, first_last, bits, out, st);
        else if (!r.u)
            e = dcmt::kitti_run(gt.u, gt.pitch, gt.fstride, r.f, r.pitch, r.fstride, rows, cols, n_frames, partials, first_last, bits, out, st);
        else
            e = dcmt::kitti_run(gt.u, gt.pitch, gt.fstride, r.u, r.pitch, r.fstride, rows, cols, n_frames, partials, first_last, bits, out, st);
        API_CUDA(e, "KITTI evaluation launch");
        return DCMT_OK;
    }
};

// `mode` is the mask of the reductions; the KITTI figures have the fixed mask g > 0 and pass DCMT_EVAL_GT_VALID
int run_evaluation(InDesc gt, InDesc r, int rows, int cols, int n_frames, int mode, void* results, void* cuda_stream, const EvalKind& kind) {
    size_t gt_span = 0, r_span = 0;
    int rc = validate_evaluation(&gt, &r, rows, cols, n_frames, mode, results, &gt_span, &r_span);
    if (rc) return rc;
    if (n_frames == 0) return DCMT_OK;
    if ((rc = check_device())) return rc;
    return kind.enqueue(gt, r, rows, cols, n_frames, results, static_cast<cudaStream_t>(cuda_stream));
}

// host pointers: both planes are staged whole (each side's own span, so 2 B/px for a uint16 side), evaluated on the
// staging copies with the caller's geometry, and the records copied back
int run_evaluation_host(InDesc gt, InDesc r, int rows, int cols, int n_frames, int mode, void* results, const EvalKind& kind) {
    size_t gt_span = 0, r_span = 0;
    int rc = validate_evaluation(&gt, &r, rows, cols, n_frames, mode, results, &gt_span, &r_span);
    if (rc) return rc;
    if (n_frames == 0) return DCMT_OK;
    const size_t res_bytes = (size_t)n_frames * kind.rec_bytes;
    Staged sg{gt.ptr(), nullptr, gt_span, gt_span, 1}, sr{r.ptr(), nullptr, r_span, r_span, 1}, sres{nullptr, results, res_bytes, res_bytes, 1};
    return run_staged({&sg, &sr, &sres}, [&](cudaStream_t st) {
        InDesc dgt = gt, dr = r;
        if (gt.u) dgt.u = static_cast<const uint16_t*>(sg.dev);
        else dgt.f = static_cast<const float*>(sg.dev);
        if (r.u) dr.u = static_cast<const uint16_t*>(sr.dev);
        else dr.f = static_cast<const float*>(sr.dev);
        return kind.enqueue(dgt, dr, rows, cols, n_frames, sres.dev, st);
    });
}

InDesc eval_f32(const float* p, size_t pitch_bytes, size_t fstride_bytes) {
    InDesc d;
    d.f = p;
    d.pitch = pitch_bytes;
    d.fstride = fstride_bytes;
    return d;
}
InDesc eval_u16(const uint16_t* p, size_t pitch_bytes, size_t fstride_bytes) {
    InDesc d;
    d.u = p;
    d.pitch = pitch_bytes;
    d.fstride = fstride_bytes;
    return d;
}

}  // namespace

extern "C" {

int dcmt_version(void) { return DCMT_VERSION; }
const char* dcmt_build_info(void) {
#ifdef DCMT_EMU
    return "emulator (tests only)";
#else
    return "cuda sm_100a";
#endif
}
const char* dcmt_last_error(void) { return g_err; }

const char* dcmt_status_string(int status) {
    switch (status) {
        case DCMT_OK: return "ok";
        case DCMT_E_BADARG: return "bad argument";
        case DCMT_E_UNSUPPORTED: return "unsupported";
        case DCMT_E_CUDA: return "CUDA error";
        case DCMT_E_NOMEM: return "out of device memory";
        default: return "unknown status";
    }
}

int dcmt_device_count(void) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) return cuda_fail(e, "cudaGetDeviceCount");
    return n;
}

int dcmt_release_workspaces(void) {
    std::lock_guard<std::mutex> lk(g_mu);
    cudaDeviceSynchronize();
    for (auto& kv : g_arenas)
        if (kv.second.base) cudaFree(kv.second.base);
    g_arenas.clear();
    return DCMT_OK;
}

size_t dcmt_workspace_bytes(int rows, int cols, int n_frames) {
    if (rows < 1 || cols < 1 || n_frames < 1) return 0;
    // upper bound over the paths a call may take: fused chunks, bilateral scratch, the guided front and the dictionary
    const int chunk = chunk_frames(rows, cols, n_frames, true);
    Arena count;
    count.counting = true;
    carve_fused(&count, rows, cols, chunk, true, true, carve_generic(&count, rows, cols, chunk, true));
    return count.used;
}

int dcmt_profile_begin(void) {
    std::lock_guard<std::mutex> lk(g_mu);
    g_prof_events.clear();
    g_prof_on = true;
    return DCMT_OK;
}

int dcmt_profile_end(double* front_ms, double* tail_ms, long long* chunks) {
    std::vector<ProfEvents> ev;
    {
        std::lock_guard<std::mutex> lk(g_mu);
        g_prof_on = false;
        ev.swap(g_prof_events);
    }
    double f = 0.0, t = 0.0;
    for (auto& pe : ev) {
        API_CUDA(cudaEventSynchronize(pe.e[2]), "profiling event");
        float a = 0.f, b = 0.f;
        API_CUDA(cudaEventElapsedTime(&a, pe.e[0], pe.e[1]), "profiling event");
        API_CUDA(cudaEventElapsedTime(&b, pe.e[1], pe.e[2]), "profiling event");
        f += a;
        t += b;
        for (int i = 0; i < 3; ++i) cudaEventDestroy(pe.e[i]);
    }
    if (front_ms) *front_ms = f;
    if (tail_ms) *tail_ms = t;
    if (chunks) *chunks = (long long)ev.size();
    return DCMT_OK;
}

int dcmt_host_alloc(size_t bytes, int write_combined, void** out) {
    if (!out || bytes == 0) return fail(DCMT_E_BADARG, "null pointer or zero size");
    int rc = check_device();
    if (rc) return rc;
    void* p = nullptr;
    cudaError_t e = cudaHostAlloc(&p, bytes, write_combined ? cudaHostAllocWriteCombined : cudaHostAllocDefault);
    if (e != cudaSuccess) return fail(DCMT_E_NOMEM, "page-locked host buffer of %zu bytes: %s", bytes, cudaGetErrorString(e));
    *out = p;
    return DCMT_OK;
}

int dcmt_host_free(void* p) {
    if (p) cudaFreeHost(p);
    return DCMT_OK;
}

long long dcmt_launch_count(void) { return dcmt::g_launches.load(std::memory_order_relaxed); }

int dcmt_img_completion_f32(const float* sparse, float* dense, int rows, int cols, size_t pitch_bytes,
                            size_t frame_stride_bytes, int n_frames, int blur_type, int flags, int32_t* stats,
                            void* cuda_stream) {
    return run_completion({nullptr, 0, false, rows, cols, blur_type, flags}, {sparse, nullptr, pitch_bytes, frame_stride_bytes},
                          {dense, nullptr, pitch_bytes, frame_stride_bytes}, n_frames, stats, static_cast<cudaStream_t>(cuda_stream));
}

int dcmt_img_completion_f32_host(const float* sparse, float* dense, int rows, int cols, size_t pitch_bytes,
                                 size_t frame_stride_bytes, int n_frames, int blur_type, int flags, int32_t* stats) {
    return run_completion_host({nullptr, 0, false, rows, cols, blur_type, flags}, {sparse, nullptr, pitch_bytes, frame_stride_bytes},
                               {dense, nullptr, pitch_bytes, frame_stride_bytes}, n_frames, stats);
}

int dcmt_img_completion_u16(const uint16_t* sparse_u16, float* dense, int rows, int cols, size_t in_pitch_bytes,
                            size_t in_frame_stride_bytes, size_t out_pitch_bytes, size_t out_frame_stride_bytes, int n_frames,
                            int blur_type, int flags, int32_t* stats, void* cuda_stream) {
    return run_completion({nullptr, 0, false, rows, cols, blur_type, flags}, {nullptr, sparse_u16, in_pitch_bytes, in_frame_stride_bytes},
                          {dense, nullptr, out_pitch_bytes, out_frame_stride_bytes}, n_frames, stats, static_cast<cudaStream_t>(cuda_stream));
}

int dcmt_img_completion_u16_host(const uint16_t* sparse_u16, float* dense, int rows, int cols, size_t in_pitch_bytes,
                                 size_t in_frame_stride_bytes, size_t out_pitch_bytes, size_t out_frame_stride_bytes,
                                 int n_frames, int blur_type, int flags, int32_t* stats) {
    return run_completion_host({nullptr, 0, false, rows, cols, blur_type, flags}, {nullptr, sparse_u16, in_pitch_bytes, in_frame_stride_bytes},
                               {dense, nullptr, out_pitch_bytes, out_frame_stride_bytes}, n_frames, stats);
}

int dcmt_img_completion_f32_host_multi(const float* sparse, float* dense, int rows, int cols, size_t pitch_bytes,
                                       size_t frame_stride_bytes, int n_frames, int blur_type, int flags, int32_t* stats,
                                       const int* devices, int n_devices) {
    return run_completion_host({nullptr, 0, false, rows, cols, blur_type, flags}, {sparse, nullptr, pitch_bytes, frame_stride_bytes},
                               {dense, nullptr, pitch_bytes, frame_stride_bytes}, n_frames, stats, devices, n_devices, true);
}

int dcmt_img_completion_u16_host_multi(const uint16_t* sparse_u16, float* dense, int rows, int cols, size_t in_pitch_bytes,
                                       size_t in_frame_stride_bytes, size_t out_pitch_bytes, size_t out_frame_stride_bytes,
                                       int n_frames, int blur_type, int flags, int32_t* stats, const int* devices, int n_devices) {
    return run_completion_host({nullptr, 0, false, rows, cols, blur_type, flags}, {nullptr, sparse_u16, in_pitch_bytes, in_frame_stride_bytes},
                               {dense, nullptr, out_pitch_bytes, out_frame_stride_bytes}, n_frames, stats, devices, n_devices, true);
}

int dcmt_img_completion_u16_u16(const uint16_t* sparse_u16, uint16_t* dense_u16, int rows, int cols, size_t in_pitch_bytes,
                                size_t in_frame_stride_bytes, size_t out_pitch_bytes, size_t out_frame_stride_bytes, int n_frames,
                                int blur_type, int flags, int32_t* stats, void* cuda_stream) {
    return run_completion({nullptr, 0, false, rows, cols, blur_type, flags}, {nullptr, sparse_u16, in_pitch_bytes, in_frame_stride_bytes},
                          {nullptr, dense_u16, out_pitch_bytes, out_frame_stride_bytes}, n_frames, stats, static_cast<cudaStream_t>(cuda_stream));
}

int dcmt_img_completion_u16_u16_host(const uint16_t* sparse_u16, uint16_t* dense_u16, int rows, int cols, size_t in_pitch_bytes,
                                     size_t in_frame_stride_bytes, size_t out_pitch_bytes, size_t out_frame_stride_bytes,
                                     int n_frames, int blur_type, int flags, int32_t* stats) {
    return run_completion_host({nullptr, 0, false, rows, cols, blur_type, flags}, {nullptr, sparse_u16, in_pitch_bytes, in_frame_stride_bytes},
                               {nullptr, dense_u16, out_pitch_bytes, out_frame_stride_bytes}, n_frames, stats);
}

int dcmt_img_completion_u16_u16_host_multi(const uint16_t* sparse_u16, uint16_t* dense_u16, int rows, int cols, size_t in_pitch_bytes,
                                           size_t in_frame_stride_bytes, size_t out_pitch_bytes, size_t out_frame_stride_bytes,
                                           int n_frames, int blur_type, int flags, int32_t* stats, const int* devices, int n_devices) {
    return run_completion_host({nullptr, 0, false, rows, cols, blur_type, flags}, {nullptr, sparse_u16, in_pitch_bytes, in_frame_stride_bytes},
                               {nullptr, dense_u16, out_pitch_bytes, out_frame_stride_bytes}, n_frames, stats, devices, n_devices, true);
}

// (a2) on KITTI uint16 input; the blur is unconditionally Gaussian in the reference (img_completion_lc.cpp:183-192)
int dcmt_interpolate_with_superpixels_u16(const uint16_t* sparse_u16, const int32_t* labels, int n_clusters, float* dense, int rows,
                                          int cols, size_t in_pitch_bytes, size_t in_frame_stride_bytes, size_t out_pitch_bytes,
                                          size_t out_frame_stride_bytes, int n_frames, int use_superpixel, int flags, int32_t* stats,
                                          void* cuda_stream) {
    return run_completion({labels, n_clusters, use_superpixel != 0, rows, cols, DCMT_BLUR_GAUSSIAN, flags},
                          {nullptr, sparse_u16, in_pitch_bytes, in_frame_stride_bytes}, {dense, nullptr, out_pitch_bytes, out_frame_stride_bytes},
                          n_frames, stats, static_cast<cudaStream_t>(cuda_stream));
}

int dcmt_interpolate_with_superpixels_u16_host(const uint16_t* sparse_u16, const int32_t* labels, int n_clusters, float* dense, int rows,
                                               int cols, size_t in_pitch_bytes, size_t in_frame_stride_bytes, size_t out_pitch_bytes,
                                               size_t out_frame_stride_bytes, int n_frames, int use_superpixel, int flags,
                                               int32_t* stats) {
    return run_completion_host({labels, n_clusters, use_superpixel != 0, rows, cols, DCMT_BLUR_GAUSSIAN, flags},
                               {nullptr, sparse_u16, in_pitch_bytes, in_frame_stride_bytes},
                               {dense, nullptr, out_pitch_bytes, out_frame_stride_bytes}, n_frames, stats);
}

int dcmt_interpolate_with_superpixels_u16_host_multi(const uint16_t* sparse_u16, const int32_t* labels, int n_clusters, float* dense,
                                                     int rows, int cols, size_t in_pitch_bytes, size_t in_frame_stride_bytes,
                                                     size_t out_pitch_bytes, size_t out_frame_stride_bytes, int n_frames,
                                                     int use_superpixel, int flags, int32_t* stats, const int* devices, int n_devices) {
    return run_completion_host({labels, n_clusters, use_superpixel != 0, rows, cols, DCMT_BLUR_GAUSSIAN, flags},
                               {nullptr, sparse_u16, in_pitch_bytes, in_frame_stride_bytes},
                               {dense, nullptr, out_pitch_bytes, out_frame_stride_bytes}, n_frames, stats, devices, n_devices, true);
}

int dcmt_interpolate_with_superpixels_u16_u16(const uint16_t* sparse_u16, const int32_t* labels, int n_clusters, uint16_t* dense_u16,
                                              int rows, int cols, size_t in_pitch_bytes, size_t in_frame_stride_bytes,
                                              size_t out_pitch_bytes, size_t out_frame_stride_bytes, int n_frames, int use_superpixel,
                                              int flags, int32_t* stats, void* cuda_stream) {
    return run_completion({labels, n_clusters, use_superpixel != 0, rows, cols, DCMT_BLUR_GAUSSIAN, flags},
                          {nullptr, sparse_u16, in_pitch_bytes, in_frame_stride_bytes},
                          {nullptr, dense_u16, out_pitch_bytes, out_frame_stride_bytes}, n_frames, stats, static_cast<cudaStream_t>(cuda_stream));
}

int dcmt_interpolate_with_superpixels_u16_u16_host(const uint16_t* sparse_u16, const int32_t* labels, int n_clusters,
                                                   uint16_t* dense_u16, int rows, int cols, size_t in_pitch_bytes,
                                                   size_t in_frame_stride_bytes, size_t out_pitch_bytes, size_t out_frame_stride_bytes,
                                                   int n_frames, int use_superpixel, int flags, int32_t* stats) {
    return run_completion_host({labels, n_clusters, use_superpixel != 0, rows, cols, DCMT_BLUR_GAUSSIAN, flags},
                               {nullptr, sparse_u16, in_pitch_bytes, in_frame_stride_bytes},
                               {nullptr, dense_u16, out_pitch_bytes, out_frame_stride_bytes}, n_frames, stats);
}

int dcmt_interpolate_with_superpixels_u16_u16_host_multi(const uint16_t* sparse_u16, const int32_t* labels, int n_clusters,
                                                         uint16_t* dense_u16, int rows, int cols, size_t in_pitch_bytes,
                                                         size_t in_frame_stride_bytes, size_t out_pitch_bytes,
                                                         size_t out_frame_stride_bytes, int n_frames, int use_superpixel, int flags,
                                                         int32_t* stats, const int* devices, int n_devices) {
    return run_completion_host({labels, n_clusters, use_superpixel != 0, rows, cols, DCMT_BLUR_GAUSSIAN, flags},
                               {nullptr, sparse_u16, in_pitch_bytes, in_frame_stride_bytes},
                               {nullptr, dense_u16, out_pitch_bytes, out_frame_stride_bytes}, n_frames, stats, devices, n_devices, true);
}

// main_lc.cpp:159-220 from the BGR frame: cvtColor(COLOR_BGR2Lab), generate_superpixels and interpolate_with_superpixels of
// KITTI uint16 depth; the Lab frames and the labels stay in the workspace
int dcmt_interpolate_with_superpixels_bgr_u16(const uint8_t* bgr, size_t bgr_pitch_bytes, size_t bgr_frame_stride_bytes,
                                              const uint16_t* sparse_u16, float* dense, int rows, int cols, size_t in_pitch_bytes,
                                              size_t in_frame_stride_bytes, size_t out_pitch_bytes, size_t out_frame_stride_bytes,
                                              int n_frames, int step, int nc, int iterations, int use_superpixel, int flags, int32_t* stats,
                                              void* cuda_stream) {
    BgrFront fr{bgr, bgr_pitch_bytes, bgr_frame_stride_bytes, step, nc, iterations};
    return run_completion_bgr({nullptr, 0, use_superpixel != 0, rows, cols, DCMT_BLUR_GAUSSIAN, flags, &fr},
                              {nullptr, sparse_u16, in_pitch_bytes, in_frame_stride_bytes},
                              {dense, nullptr, out_pitch_bytes, out_frame_stride_bytes}, n_frames, stats, static_cast<cudaStream_t>(cuda_stream));
}

int dcmt_interpolate_with_superpixels_bgr_u16_host(const uint8_t* bgr, size_t bgr_pitch_bytes, size_t bgr_frame_stride_bytes,
                                                   const uint16_t* sparse_u16, float* dense, int rows, int cols, size_t in_pitch_bytes,
                                                   size_t in_frame_stride_bytes, size_t out_pitch_bytes, size_t out_frame_stride_bytes,
                                                   int n_frames, int step, int nc, int iterations, int use_superpixel, int flags,
                                                   int32_t* stats) {
    BgrFront fr{bgr, bgr_pitch_bytes, bgr_frame_stride_bytes, step, nc, iterations};
    return run_completion_host({nullptr, 0, use_superpixel != 0, rows, cols, DCMT_BLUR_GAUSSIAN, flags, &fr},
                               {nullptr, sparse_u16, in_pitch_bytes, in_frame_stride_bytes},
                               {dense, nullptr, out_pitch_bytes, out_frame_stride_bytes}, n_frames, stats);
}

int dcmt_interpolate_with_superpixels_bgr_u16_host_multi(const uint8_t* bgr, size_t bgr_pitch_bytes, size_t bgr_frame_stride_bytes,
                                                         const uint16_t* sparse_u16, float* dense, int rows, int cols, size_t in_pitch_bytes,
                                                         size_t in_frame_stride_bytes, size_t out_pitch_bytes, size_t out_frame_stride_bytes,
                                                         int n_frames, int step, int nc, int iterations, int use_superpixel, int flags,
                                                         int32_t* stats, const int* devices, int n_devices) {
    BgrFront fr{bgr, bgr_pitch_bytes, bgr_frame_stride_bytes, step, nc, iterations};
    return run_completion_host({nullptr, 0, use_superpixel != 0, rows, cols, DCMT_BLUR_GAUSSIAN, flags, &fr},
                               {nullptr, sparse_u16, in_pitch_bytes, in_frame_stride_bytes},
                               {dense, nullptr, out_pitch_bytes, out_frame_stride_bytes}, n_frames, stats, devices, n_devices, true);
}

int dcmt_interpolate_with_superpixels_bgr_u16_u16(const uint8_t* bgr, size_t bgr_pitch_bytes, size_t bgr_frame_stride_bytes,
                                                  const uint16_t* sparse_u16, uint16_t* dense_u16, int rows, int cols, size_t in_pitch_bytes,
                                                  size_t in_frame_stride_bytes, size_t out_pitch_bytes, size_t out_frame_stride_bytes,
                                                  int n_frames, int step, int nc, int iterations, int use_superpixel, int flags,
                                                  int32_t* stats, void* cuda_stream) {
    BgrFront fr{bgr, bgr_pitch_bytes, bgr_frame_stride_bytes, step, nc, iterations};
    return run_completion_bgr({nullptr, 0, use_superpixel != 0, rows, cols, DCMT_BLUR_GAUSSIAN, flags, &fr},
                              {nullptr, sparse_u16, in_pitch_bytes, in_frame_stride_bytes},
                              {nullptr, dense_u16, out_pitch_bytes, out_frame_stride_bytes}, n_frames, stats,
                              static_cast<cudaStream_t>(cuda_stream));
}

int dcmt_interpolate_with_superpixels_bgr_u16_u16_host(const uint8_t* bgr, size_t bgr_pitch_bytes, size_t bgr_frame_stride_bytes,
                                                       const uint16_t* sparse_u16, uint16_t* dense_u16, int rows, int cols,
                                                       size_t in_pitch_bytes, size_t in_frame_stride_bytes, size_t out_pitch_bytes,
                                                       size_t out_frame_stride_bytes, int n_frames, int step, int nc, int iterations,
                                                       int use_superpixel, int flags, int32_t* stats) {
    BgrFront fr{bgr, bgr_pitch_bytes, bgr_frame_stride_bytes, step, nc, iterations};
    return run_completion_host({nullptr, 0, use_superpixel != 0, rows, cols, DCMT_BLUR_GAUSSIAN, flags, &fr},
                               {nullptr, sparse_u16, in_pitch_bytes, in_frame_stride_bytes},
                               {nullptr, dense_u16, out_pitch_bytes, out_frame_stride_bytes}, n_frames, stats);
}

int dcmt_interpolate_with_superpixels_bgr_u16_u16_host_multi(const uint8_t* bgr, size_t bgr_pitch_bytes, size_t bgr_frame_stride_bytes,
                                                             const uint16_t* sparse_u16, uint16_t* dense_u16, int rows, int cols,
                                                             size_t in_pitch_bytes, size_t in_frame_stride_bytes, size_t out_pitch_bytes,
                                                             size_t out_frame_stride_bytes, int n_frames, int step, int nc, int iterations,
                                                             int use_superpixel, int flags, int32_t* stats, const int* devices,
                                                             int n_devices) {
    BgrFront fr{bgr, bgr_pitch_bytes, bgr_frame_stride_bytes, step, nc, iterations};
    return run_completion_host({nullptr, 0, use_superpixel != 0, rows, cols, DCMT_BLUR_GAUSSIAN, flags, &fr},
                               {nullptr, sparse_u16, in_pitch_bytes, in_frame_stride_bytes},
                               {nullptr, dense_u16, out_pitch_bytes, out_frame_stride_bytes}, n_frames, stats, devices, n_devices, true);
}

int dcmt_depth_to_u16(const float* depth, uint16_t* out, int rows, int cols, size_t in_pitch_bytes, size_t in_frame_stride_bytes,
                      size_t out_pitch_bytes, size_t out_frame_stride_bytes, int n_frames, void* cuda_stream) {
    if (!depth || !out) return fail(DCMT_E_BADARG, "null image pointer");
    Geometry gi, go;
    int rc = check_geometry(rows, cols, in_pitch_bytes, in_frame_stride_bytes, n_frames, &gi, sizeof(float));
    if (rc) return rc;
    if ((rc = check_geometry(rows, cols, out_pitch_bytes, out_frame_stride_bytes, n_frames, &go, sizeof(uint16_t)))) return rc;
    if (n_frames && overlaps(depth, gi.span_bytes, out, go.span_bytes)) return fail(DCMT_E_BADARG, "input and output overlap");
    if (n_frames == 0) return DCMT_OK;
    if ((rc = check_device())) return rc;
    API_CUDA(dcmt::depth_to_u16(depth, gi.pitch, gi.fstride, out, go.pitch, go.fstride, rows, cols, n_frames,
                                static_cast<cudaStream_t>(cuda_stream)),
             "uint16 conversion launch");
    return DCMT_OK;
}

int dcmt_interpolate_with_superpixels_f32_host_multi(const float* sparse, const int32_t* labels, int n_clusters, float* dense, int rows,
                                                     int cols, size_t pitch_bytes, size_t frame_stride_bytes, int n_frames,
                                                     int use_superpixel, int flags, int32_t* stats, const int* devices, int n_devices) {
    return run_completion_host({labels, n_clusters, use_superpixel != 0, rows, cols, DCMT_BLUR_GAUSSIAN, flags},
                               {sparse, nullptr, pitch_bytes, frame_stride_bytes}, {dense, nullptr, pitch_bytes, frame_stride_bytes},
                               n_frames, stats, devices, n_devices, true);
}

int dcmt_debug_host_copy_f32(const float* in, float* out, int rows, int cols, int n_frames, const int* devices, int n_devices) {
    return run_completion_host({nullptr, 0, false, rows, cols, DCMT_BLUR_NONE, DCMT_PATH_AUTO}, {in}, {out}, n_frames, nullptr, devices,
                               n_devices, devices != nullptr || n_devices != 0, true);
}

int dcmt_debug_host_copy_u16(const uint16_t* in, float* out, int rows, int cols, int n_frames, const int* devices, int n_devices) {
    return run_completion_host({nullptr, 0, false, rows, cols, DCMT_BLUR_NONE, DCMT_PATH_AUTO}, {nullptr, in}, {out}, n_frames, nullptr,
                               devices, n_devices, devices != nullptr || n_devices != 0, true);
}

int dcmt_debug_host_copy_u16_u16(const uint16_t* in, uint16_t* out, int rows, int cols, int n_frames, const int* devices, int n_devices) {
    return run_completion_host({nullptr, 0, false, rows, cols, DCMT_BLUR_NONE, DCMT_PATH_AUTO}, {nullptr, in}, {nullptr, out}, n_frames,
                               nullptr, devices, n_devices, devices != nullptr || n_devices != 0, true);
}

int dcmt_interpolate_with_superpixels_ex_f32(const float* sparse, const int32_t* labels, int n_clusters, float* dense, int rows,
                                             int cols, size_t pitch_bytes, size_t frame_stride_bytes, int n_frames, int use_superpixel,
                                             int flags, int32_t* stats, void* cuda_stream) {
    // blur is unconditionally Gaussian in the reference (img_completion_lc.cpp:183-192)
    return run_completion({labels, n_clusters, use_superpixel != 0, rows, cols, DCMT_BLUR_GAUSSIAN, flags},
                          {sparse, nullptr, pitch_bytes, frame_stride_bytes}, {dense, nullptr, pitch_bytes, frame_stride_bytes}, n_frames,
                          stats, static_cast<cudaStream_t>(cuda_stream));
}

int dcmt_interpolate_with_superpixels_ex_f32_host(const float* sparse, const int32_t* labels, int n_clusters, float* dense, int rows,
                                                  int cols, size_t pitch_bytes, size_t frame_stride_bytes, int n_frames,
                                                  int use_superpixel, int flags, int32_t* stats) {
    return run_completion_host({labels, n_clusters, use_superpixel != 0, rows, cols, DCMT_BLUR_GAUSSIAN, flags},
                               {sparse, nullptr, pitch_bytes, frame_stride_bytes}, {dense, nullptr, pitch_bytes, frame_stride_bytes},
                               n_frames, stats);
}

int dcmt_interpolate_with_superpixels_f32(const float* sparse, const int32_t* labels, int n_clusters, float* dense,
                                          int rows, int cols, size_t pitch_bytes, size_t frame_stride_bytes, int n_frames,
                                          int use_superpixel, int32_t* stats, void* cuda_stream) {
    return dcmt_interpolate_with_superpixels_ex_f32(sparse, labels, n_clusters, dense, rows, cols, pitch_bytes, frame_stride_bytes,
                                                    n_frames, use_superpixel, DCMT_PATH_AUTO, stats, cuda_stream);
}

int dcmt_interpolate_with_superpixels_f32_host(const float* sparse, const int32_t* labels, int n_clusters, float* dense,
                                               int rows, int cols, size_t pitch_bytes, size_t frame_stride_bytes,
                                               int n_frames, int use_superpixel, int32_t* stats) {
    return dcmt_interpolate_with_superpixels_ex_f32_host(sparse, labels, n_clusters, dense, rows, cols, pitch_bytes,
                                                         frame_stride_bytes, n_frames, use_superpixel, DCMT_PATH_AUTO, stats);
}

int dcmt_img_completion_stages_f32(const float* sparse, float* dense, int rows, int cols, int blur_type, float* stages,
                                   int n_stages, uint32_t* stage_mask_out, void* cuda_stream) {
    if (!stages || n_stages < dcmt::kOracleStages) return fail(DCMT_E_BADARG, "stages buffer must hold %d planes", dcmt::kOracleStages);
    uint32_t mask = 0;
    int rc = run_completion({nullptr, 0, false, rows, cols, blur_type, DCMT_PATH_GENERIC}, {sparse}, {dense}, 1, nullptr,
                            static_cast<cudaStream_t>(cuda_stream), stages, &mask);
    if (stage_mask_out) *stage_mask_out = mask;
    return rc;
}

int dcmt_debug_q8_phase_cycles(const float* sparse, float* dense, int rows, int cols, int n_frames, long long* front_stamps,
                               long long* tail_stamps, int* tiles_per_frame, void* cuda_stream) {
    // debugging aid: the fused kernels on one chunk with per-CTA clock64() stamps at the phase boundaries
    if (!sparse || !dense || rows < dcmt::kQ8MinRows || cols < dcmt::kQ8MinCols || n_frames < 1) return fail(DCMT_E_BADARG, "bad argument");
    int rc = check_device();
    if (rc) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    API_CUDA(dcmt::q8_configure(), "kernel attribute setup");
    CompletionCall cc{nullptr, 0, false, rows, cols, DCMT_BLUR_GAUSSIAN, DCMT_PATH_AUTO};
    if (!fused_applies(cc)) return fail(DCMT_E_UNSUPPORTED, "shape not served by the fused kernels");
    const size_t fpix = (size_t)rows * cols;
    dcmt::Q8Plan p{};
    if ((rc = acquire_carved(st, [&](Arena* a) { p = carve_fused(a, rows, cols, n_frames, false, false, carve_generic(a, rows, cols, n_frames, false)).p; })))
        return rc;
    p.prof_front = front_stamps;
    p.prof_tail = tail_stamps;
    if (tiles_per_frame) *tiles_per_frame = ((cols + p.tw - 1) / p.tw) * ((rows + p.th - 1) / p.th);
    API_CUDA(dcmt::q8_run_front(p, sparse, nullptr, cols, fpix, n_frames, 1, st), "fused front launch");
    API_CUDA(dcmt::q8_run_tail(p, dense, nullptr, cols, fpix, n_frames, DCMT_BLUR_GAUSSIAN, st), "fused tail launch");
    return DCMT_OK;
}

int dcmt_slic_center_count(int rows, int cols, int step) {
    if (rows < 1 || cols < 1 || step < 1) return 0;
    return dcmt::slic_center_count(rows, cols, step);
}

static int check_slic_call(const uint8_t* img, const int32_t* labels, int rows, int cols, int n_frames, int step, int nc, int iterations) {
    if (!img || !labels) return fail(DCMT_E_BADARG, "null pointer");
    int rc = check_planes(rows, cols, n_frames);
    if (rc) return rc;
    if ((rc = check_slic(rows, cols, step, nc, iterations))) return rc;
    if ((size_t)rows * (size_t)cols > (size_t)1 << 30) return fail(DCMT_E_UNSUPPORTED, "frame larger than 2^30 pixels");
    if (n_frames > 65535) return fail(DCMT_E_UNSUPPORTED, "at most 65535 frames per call");
    return DCMT_OK;
}

// Slic::generate_superpixels on the Lab image `img`, or, with from_bgr, on the cvtColor(COLOR_BGR2Lab) of the BGR image
// `img`: the Lab frames then live in the SLIC workspace of (device, stream) and never leave the device
static int slic_device(const uint8_t* img, bool from_bgr, int rows, int cols, int n_frames, int step, int nc, int iterations,
                       int32_t* labels, double* centers, void* cuda_stream) {
    int rc = check_slic_call(img, labels, rows, cols, n_frames, step, nc, iterations);
    if (rc) return rc;
    if (n_frames == 0) return DCMT_OK;
    if ((rc = check_device())) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    SlicBuffers s;
    if ((rc = acquire_carved(st, [&](Arena* a) { s = carve_slic(a, rows, cols, n_frames, step, from_bgr); }))) return rc;
    const size_t pitch = (size_t)cols * 3;
    return enqueue_slic(s, img, pitch, pitch * rows, from_bgr, rows, cols, n_frames, step, nc, iterations, labels, centers, st);
}

int dcmt_slic_u8c3(const uint8_t* lab, int rows, int cols, int n_frames, int step, int nc, int iterations, int32_t* labels,
                   double* centers, void* cuda_stream) {
    return slic_device(lab, false, rows, cols, n_frames, step, nc, iterations, labels, centers, cuda_stream);
}

int dcmt_slic_bgr_u8c3(const uint8_t* bgr, int rows, int cols, int n_frames, int step, int nc, int iterations, int32_t* labels,
                       double* centers, void* cuda_stream) {
    return slic_device(bgr, true, rows, cols, n_frames, step, nc, iterations, labels, centers, cuda_stream);
}

static int slic_host(const uint8_t* img, bool from_bgr, int rows, int cols, int n_frames, int step, int nc, int iterations,
                     int32_t* labels, double* centers) {
    int rc = check_slic_call(img, labels, rows, cols, n_frames, step, nc, iterations);
    if (rc) return rc;
    if (n_frames == 0) return DCMT_OK;
    const size_t n = (size_t)rows * cols * n_frames;
    const size_t kb = (size_t)dcmt::slic_center_count(rows, cols, step) * n_frames * 5 * sizeof(double);
    Staged si{img, nullptr, n * 3, n * 3, 1}, sl{nullptr, labels, n * 4, n * 4, 1}, sc{nullptr, kb ? centers : nullptr, kb, kb, 1};
    return run_staged({&si, &sl, &sc}, [&](cudaStream_t st) {
        SlicBuffers s;
        if (int rc2 = acquire_carved(st, [&](Arena* a) { s = carve_slic(a, rows, cols, n_frames, step, from_bgr); })) return rc2;
        const size_t pitch = (size_t)cols * 3;
        return enqueue_slic(s, static_cast<const uint8_t*>(si.dev), pitch, pitch * rows, from_bgr, rows, cols, n_frames, step, nc, iterations,
                            static_cast<int32_t*>(sl.dev), centers ? static_cast<double*>(sc.dev) : nullptr, st);
    });
}

int dcmt_slic_u8c3_host(const uint8_t* lab, int rows, int cols, int n_frames, int step, int nc, int iterations, int32_t* labels,
                        double* centers) {
    return slic_host(lab, false, rows, cols, n_frames, step, nc, iterations, labels, centers);
}

int dcmt_slic_bgr_u8c3_host(const uint8_t* bgr, int rows, int cols, int n_frames, int step, int nc, int iterations, int32_t* labels,
                            double* centers) {
    return slic_host(bgr, true, rows, cols, n_frames, step, nc, iterations, labels, centers);
}

static int check_project(const float* points, int n_points, const float* T_host, const float* P_host, int rows, int cols) {
    if ((!points && n_points > 0) || !T_host || !P_host) return fail(DCMT_E_BADARG, "null pointer");
    if (n_points < 0) return fail(DCMT_E_BADARG, "n_points must be >= 0 (got %d)", n_points);
    int rc = check_planes(rows, cols, 1);
    if (rc) return rc;
    if ((size_t)rows * (size_t)cols > (size_t)1 << 30) return fail(DCMT_E_UNSUPPORTED, "frame larger than 2^30 pixels");
    return DCMT_OK;
}

// the projection on validated arguments, 16-byte aligned points: its keys and counters in the stream's arena
static int enqueue_project(const float* points, int n_points, const float* T_host, const float* P_host, int rows, int cols,
                           float* projected, float* normalized, float norm_a, float norm_b, int32_t* n_projected, cudaStream_t st) {
    dcmt::ProjectWork w{};
    if (int rc = acquire_carved(st, [&](Arena* a) { w = carve_project(a, rows, cols, 1); })) return rc;
    return enqueue_project_batch(w, points, nullptr, n_points, 0, 1, T_host, P_host, rows, cols, projected, normalized, norm_a, norm_b, n_projected,
                                 st);
}

int dcmt_lidar_project_f32(const float* points, int n_points, const float* T_host, const float* P_host, int rows, int cols,
                           float* projected, float* normalized, float norm_a, float norm_b, int32_t* n_projected, void* cuda_stream) {
    int rc = check_project(points, n_points, T_host, P_host, rows, cols);
    if (rc) return rc;
    if (points && (reinterpret_cast<uintptr_t>(points) & 15)) return fail(DCMT_E_BADARG, "points must be 16-byte aligned");
    if ((rc = check_device())) return rc;
    return enqueue_project(points, n_points, T_host, P_host, rows, cols, projected, normalized, norm_a, norm_b, n_projected,
                           static_cast<cudaStream_t>(cuda_stream));
}

int dcmt_lidar_project_batch_f32(const float* points, const int32_t* n_points_dev_or_null, int max_points, size_t cloud_stride_points,
                                 int n_clouds, const float* T_host, const float* P_host, int rows, int cols, float* projected,
                                 float* normalized, float norm_a, float norm_b, int32_t* n_projected, void* cuda_stream) {
    int rc = check_project_batch(points, max_points, cloud_stride_points, n_clouds, 65535, T_host, P_host, rows, cols);
    if (rc) return rc;
    if (points && (reinterpret_cast<uintptr_t>(points) & 15)) return fail(DCMT_E_BADARG, "points must be 16-byte aligned");
    if (n_clouds == 0) return DCMT_OK;
    if ((rc = check_device())) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    dcmt::ProjectWork w{};
    if ((rc = acquire_carved(st, [&](Arena* a) { w = carve_project(a, rows, cols, n_clouds); }))) return rc;
    return enqueue_project_batch(w, points, n_points_dev_or_null, max_points, cloud_stride_points, n_clouds, T_host, P_host, rows, cols, projected,
                                 normalized, norm_a, norm_b, n_projected, st);
}

int dcmt_lidar_project_f32_host(const float* points, int n_points, const float* T_host, const float* P_host, int rows, int cols,
                                float* projected, float* normalized, float norm_a, float norm_b, int32_t* n_projected) {
    int rc = check_project(points, n_points, T_host, P_host, rows, cols);
    if (rc) return rc;
    // the points are staged whole into an aligned buffer; the kernel writes every plane, copied back where the caller wants it
    const size_t pb = (size_t)n_points * 16, n = (size_t)rows * cols * 4;
    Staged sp{n_points > 0 ? points : nullptr, nullptr, pb, pb, 1}, sj{nullptr, projected, n, n, 1}, sn{nullptr, normalized, n, n, 1},
        sc{nullptr, n_projected, 4, 4, 1};
    return run_staged({&sp, &sj, &sn, &sc}, [&](cudaStream_t st) {
        return enqueue_project(static_cast<const float*>(sp.dev), n_points, T_host, P_host, rows, cols, static_cast<float*>(sj.dev),
                               static_cast<float*>(sn.dev), norm_a, norm_b, static_cast<int32_t*>(sc.dev), st);
    });
}

static_assert(sizeof(dcmt_eval_result) == sizeof(dcmt::EvalResult), "dcmt_eval_result and dcmt::EvalResult must match");

int dcmt_evaluate_f32(const float* gt, const float* dense, int rows, int cols, size_t pitch_bytes, size_t frame_stride_bytes,
                      int n_frames, float tolerance, int mode, dcmt_eval_result* results, void* cuda_stream) {
    return run_evaluation(eval_f32(gt, pitch_bytes, frame_stride_bytes), eval_f32(dense, pitch_bytes, frame_stride_bytes), rows, cols,
                          n_frames, mode, results, cuda_stream, EvalReductions(tolerance, mode));
}

int dcmt_evaluate_f32_host(const float* gt, const float* dense, int rows, int cols, size_t pitch_bytes, size_t frame_stride_bytes,
                           int n_frames, float tolerance, int mode, dcmt_eval_result* results) {
    return run_evaluation_host(eval_f32(gt, pitch_bytes, frame_stride_bytes), eval_f32(dense, pitch_bytes, frame_stride_bytes), rows, cols,
                               n_frames, mode, results, EvalReductions(tolerance, mode));
}

int dcmt_evaluate_u16(const uint16_t* gt_u16, const float* dense, int rows, int cols, size_t gt_pitch_bytes, size_t gt_frame_stride_bytes,
                      size_t dense_pitch_bytes, size_t dense_frame_stride_bytes, int n_frames, float tolerance, int mode,
                      dcmt_eval_result* results, void* cuda_stream) {
    return run_evaluation(eval_u16(gt_u16, gt_pitch_bytes, gt_frame_stride_bytes), eval_f32(dense, dense_pitch_bytes, dense_frame_stride_bytes),
                          rows, cols, n_frames, mode, results, cuda_stream, EvalReductions(tolerance, mode));
}

int dcmt_evaluate_u16_host(const uint16_t* gt_u16, const float* dense, int rows, int cols, size_t gt_pitch_bytes,
                           size_t gt_frame_stride_bytes, size_t dense_pitch_bytes, size_t dense_frame_stride_bytes, int n_frames,
                           float tolerance, int mode, dcmt_eval_result* results) {
    return run_evaluation_host(eval_u16(gt_u16, gt_pitch_bytes, gt_frame_stride_bytes),
                               eval_f32(dense, dense_pitch_bytes, dense_frame_stride_bytes), rows, cols, n_frames, mode, results,
                               EvalReductions(tolerance, mode));
}

int dcmt_evaluate_u16_u16(const uint16_t* gt_u16, const uint16_t* dense_u16, int rows, int cols, size_t gt_pitch_bytes,
                          size_t gt_frame_stride_bytes, size_t dense_pitch_bytes, size_t dense_frame_stride_bytes, int n_frames,
                          float tolerance, int mode, dcmt_eval_result* results, void* cuda_stream) {
    return run_evaluation(eval_u16(gt_u16, gt_pitch_bytes, gt_frame_stride_bytes),
                          eval_u16(dense_u16, dense_pitch_bytes, dense_frame_stride_bytes), rows, cols, n_frames, mode, results, cuda_stream,
                          EvalReductions(tolerance, mode));
}

int dcmt_evaluate_u16_u16_host(const uint16_t* gt_u16, const uint16_t* dense_u16, int rows, int cols, size_t gt_pitch_bytes,
                               size_t gt_frame_stride_bytes, size_t dense_pitch_bytes, size_t dense_frame_stride_bytes, int n_frames,
                               float tolerance, int mode, dcmt_eval_result* results) {
    return run_evaluation_host(eval_u16(gt_u16, gt_pitch_bytes, gt_frame_stride_bytes),
                               eval_u16(dense_u16, dense_pitch_bytes, dense_frame_stride_bytes), rows, cols, n_frames, mode, results,
                               EvalReductions(tolerance, mode));
}

static_assert(sizeof(dcmt_kitti_metrics) == sizeof(dcmt::KittiMetrics) && sizeof(dcmt_kitti_metrics) == 80,
              "dcmt_kitti_metrics and dcmt::KittiMetrics must match");

int dcmt_evaluate_kitti_f32(const float* gt, const float* pred, int rows, int cols, size_t gt_pitch_bytes, size_t gt_frame_stride_bytes,
                            size_t pred_pitch_bytes, size_t pred_frame_stride_bytes, int n_frames, dcmt_kitti_metrics* results,
                            void* cuda_stream) {
    return run_evaluation(eval_f32(gt, gt_pitch_bytes, gt_frame_stride_bytes), eval_f32(pred, pred_pitch_bytes, pred_frame_stride_bytes),
                          rows, cols, n_frames, DCMT_EVAL_GT_VALID, results, cuda_stream, EvalKitti());
}

int dcmt_evaluate_kitti_f32_host(const float* gt, const float* pred, int rows, int cols, size_t gt_pitch_bytes,
                                 size_t gt_frame_stride_bytes, size_t pred_pitch_bytes, size_t pred_frame_stride_bytes, int n_frames,
                                 dcmt_kitti_metrics* results) {
    return run_evaluation_host(eval_f32(gt, gt_pitch_bytes, gt_frame_stride_bytes), eval_f32(pred, pred_pitch_bytes, pred_frame_stride_bytes),
                               rows, cols, n_frames, DCMT_EVAL_GT_VALID, results, EvalKitti());
}

int dcmt_evaluate_kitti_u16(const uint16_t* gt_u16, const float* pred, int rows, int cols, size_t gt_pitch_bytes,
                            size_t gt_frame_stride_bytes, size_t pred_pitch_bytes, size_t pred_frame_stride_bytes, int n_frames,
                            dcmt_kitti_metrics* results, void* cuda_stream) {
    return run_evaluation(eval_u16(gt_u16, gt_pitch_bytes, gt_frame_stride_bytes), eval_f32(pred, pred_pitch_bytes, pred_frame_stride_bytes),
                          rows, cols, n_frames, DCMT_EVAL_GT_VALID, results, cuda_stream, EvalKitti());
}

int dcmt_evaluate_kitti_u16_host(const uint16_t* gt_u16, const float* pred, int rows, int cols, size_t gt_pitch_bytes,
                                 size_t gt_frame_stride_bytes, size_t pred_pitch_bytes, size_t pred_frame_stride_bytes, int n_frames,
                                 dcmt_kitti_metrics* results) {
    return run_evaluation_host(eval_u16(gt_u16, gt_pitch_bytes, gt_frame_stride_bytes),
                               eval_f32(pred, pred_pitch_bytes, pred_frame_stride_bytes), rows, cols, n_frames, DCMT_EVAL_GT_VALID, results,
                               EvalKitti());
}

int dcmt_evaluate_kitti_u16_u16(const uint16_t* gt_u16, const uint16_t* pred_u16, int rows, int cols, size_t gt_pitch_bytes,
                                size_t gt_frame_stride_bytes, size_t pred_pitch_bytes, size_t pred_frame_stride_bytes, int n_frames,
                                dcmt_kitti_metrics* results, void* cuda_stream) {
    return run_evaluation(eval_u16(gt_u16, gt_pitch_bytes, gt_frame_stride_bytes),
                          eval_u16(pred_u16, pred_pitch_bytes, pred_frame_stride_bytes), rows, cols, n_frames, DCMT_EVAL_GT_VALID, results,
                          cuda_stream, EvalKitti());
}

int dcmt_evaluate_kitti_u16_u16_host(const uint16_t* gt_u16, const uint16_t* pred_u16, int rows, int cols, size_t gt_pitch_bytes,
                                     size_t gt_frame_stride_bytes, size_t pred_pitch_bytes, size_t pred_frame_stride_bytes, int n_frames,
                                     dcmt_kitti_metrics* results) {
    return run_evaluation_host(eval_u16(gt_u16, gt_pitch_bytes, gt_frame_stride_bytes),
                               eval_u16(pred_u16, pred_pitch_bytes, pred_frame_stride_bytes), rows, cols, n_frames, DCMT_EVAL_GT_VALID,
                               results, EvalKitti());
}

void dcmt_stereo_params_default(dcmt_stereo_params* p) {
    if (!p) return;
    p->baseline = 0.54f;
    p->focal = 9.597910e+02f;
    p->damp_factor = 500.0f;
    p->err_clip = 255.0f;
    p->depth_clip = 100.0f;
    p->num_iterations = 4;
    p->final_gauss = 1;
}

void dcmt_stereo_params_official(dcmt_stereo_params* p, int num_iterations) {
    if (!p) return;
    dcmt_stereo_params_default(p);
    p->damp_factor = 1370.0f;
    p->err_clip = 221.0f;
    p->depth_clip = 80.0f;
    p->num_iterations = num_iterations;
    p->final_gauss = 0;
}

static int check_stereo_refine(const float* depth_ig, const uint8_t* left_gray, const uint8_t* right_gray, const float* depth_out,
                               int rows, int cols, int n_frames, const dcmt_stereo_params* prm) {
    if (!depth_ig || !left_gray || !right_gray || !depth_out || !prm) return fail(DCMT_E_BADARG, "null pointer");
    int rc = check_planes(rows, cols, n_frames);
    if (rc) return rc;
    if (prm->num_iterations < 0) return fail(DCMT_E_BADARG, "num_iterations %d", prm->num_iterations);
    if ((size_t)rows * (size_t)cols > (size_t)1 << 30) return fail(DCMT_E_UNSUPPORTED, "frame larger than 2^30 pixels");
    return DCMT_OK;
}

int dcmt_stereo_refine_f32(const float* depth_ig, const uint8_t* left_gray, const uint8_t* right_gray, float* depth_out,
                           float* disp_out, int rows, int cols, int n_frames, const dcmt_stereo_params* prm,
                           void* cuda_stream) {
    int rc = check_stereo_refine(depth_ig, left_gray, right_gray, depth_out, rows, cols, n_frames, prm);
    if (rc) return rc;
    if (n_frames == 0) return DCMT_OK;
    const size_t bytes = (size_t)rows * cols * n_frames * sizeof(float);
    if (overlaps(depth_ig, bytes, depth_out, bytes)) return fail(DCMT_E_BADARG, "input and output overlap");
    if ((rc = check_device())) return rc;
    API_CUDA(dcmt::stereo_refine(depth_ig, left_gray, right_gray, depth_out, disp_out, rows, cols, n_frames, prm->baseline,
                                 prm->focal, prm->damp_factor, prm->err_clip, prm->depth_clip, prm->num_iterations,
                                 prm->final_gauss, static_cast<cudaStream_t>(cuda_stream)),
             "stereo refine launch");
    return DCMT_OK;
}

int dcmt_stereo_refine_f32_host(const float* depth_ig, const uint8_t* left_gray, const uint8_t* right_gray,
                                float* depth_out, float* disp_out, int rows, int cols, int n_frames,
                                const dcmt_stereo_params* prm) {
    int rc = check_stereo_refine(depth_ig, left_gray, right_gray, depth_out, rows, cols, n_frames, prm);
    if (rc) return rc;
    if (n_frames == 0) return DCMT_OK;
    // one device of the host chunk pipeline: H2D -> kernel -> D2H (asynchronous for page-locked buffers)
    const size_t fpix = (size_t)rows * cols;
    auto chunk = [&](Lane&, cudaStream_t st, int f0, int nf, int hc, int) -> int {
        float *d_ig, *d_out, *d_disp;
        uint8_t *d_l, *d_r;
        int rc2 = acquire_carved(st, [&](Arena* a) {
            d_ig = carve<float>(a, fpix * hc);
            d_out = carve<float>(a, fpix * hc);
            d_disp = disp_out ? carve<float>(a, fpix * hc) : nullptr;
            d_l = carve<uint8_t>(a, fpix * hc);
            d_r = carve<uint8_t>(a, fpix * hc);
        });
        if (rc2) return rc2;
        const size_t off = (size_t)f0 * fpix, n = fpix * nf;
        API_CUDA(cudaMemcpyAsync(d_ig, depth_ig + off, n * 4, cudaMemcpyHostToDevice, st), "host to device copy");
        API_CUDA(cudaMemcpyAsync(d_l, left_gray + off, n, cudaMemcpyHostToDevice, st), "host to device copy");
        API_CUDA(cudaMemcpyAsync(d_r, right_gray + off, n, cudaMemcpyHostToDevice, st), "host to device copy");
        API_CUDA(dcmt::stereo_refine(d_ig, d_l, d_r, d_out, d_disp, rows, cols, nf, prm->baseline, prm->focal, prm->damp_factor,
                                     prm->err_clip, prm->depth_clip, prm->num_iterations, prm->final_gauss, st),
                 "stereo refine launch");
        API_CUDA(cudaMemcpyAsync(depth_out + off, d_out, n * 4, cudaMemcpyDeviceToHost, st), "device to host copy");
        if (disp_out) API_CUDA(cudaMemcpyAsync(disp_out + off, d_disp, n * 4, cudaMemcpyDeviceToHost, st), "device to host copy");
        return DCMT_OK;
    };
    return run_host_chunks(n_frames, rows, cols, nullptr, 0, false, false, false, DCMT_PATH_GENERIC, chunk);
}

int dcmt_stereo_chain_f32(const float* points, const int32_t* n_points_or_null, int max_points, size_t cloud_stride_points, const float* T_host,
                          const float* P_host, float norm_a, float norm_b, const uint8_t* left_bgr, const uint8_t* right_bgr, size_t bgr_pitch_bytes,
                          size_t bgr_frame_stride_bytes, float* depth_out, float* disp_out_or_null, int rows, int cols, int n_frames, int step,
                          int nc, int iterations, int use_superpixel, int flags, const dcmt_stereo_params* params, int32_t* stats_or_null,
                          void* cuda_stream) {
    return run_stereo_chain({points, n_points_or_null, max_points, cloud_stride_points, T_host, P_host, norm_a, norm_b, left_bgr, right_bgr,
                             bgr_pitch_bytes, bgr_frame_stride_bytes, depth_out, disp_out_or_null, rows, cols, n_frames, step, nc, iterations,
                             use_superpixel, flags, params, stats_or_null},
                            static_cast<cudaStream_t>(cuda_stream));
}

int dcmt_stereo_chain_f32_host(const float* points, const int32_t* n_points_or_null, int max_points, size_t cloud_stride_points,
                               const float* T_host, const float* P_host, float norm_a, float norm_b, const uint8_t* left_bgr,
                               const uint8_t* right_bgr, size_t bgr_pitch_bytes, size_t bgr_frame_stride_bytes, float* depth_out,
                               float* disp_out_or_null, int rows, int cols, int n_frames, int step, int nc, int iterations, int use_superpixel,
                               int flags, const dcmt_stereo_params* params, int32_t* stats_or_null) {
    return run_stereo_chain_host({points, n_points_or_null, max_points, cloud_stride_points, T_host, P_host, norm_a, norm_b, left_bgr, right_bgr,
                                  bgr_pitch_bytes, bgr_frame_stride_bytes, depth_out, disp_out_or_null, rows, cols, n_frames, step, nc,
                                  iterations, use_superpixel, flags, params, stats_or_null});
}

int dcmt_stereo_chain_f32_host_multi(const float* points, const int32_t* n_points_or_null, int max_points, size_t cloud_stride_points,
                                     const float* T_host, const float* P_host, float norm_a, float norm_b, const uint8_t* left_bgr,
                                     const uint8_t* right_bgr, size_t bgr_pitch_bytes, size_t bgr_frame_stride_bytes, float* depth_out,
                                     float* disp_out_or_null, int rows, int cols, int n_frames, int step, int nc, int iterations,
                                     int use_superpixel, int flags, const dcmt_stereo_params* params, int32_t* stats_or_null,
                                     const int* devices_or_null, int n_devices) {
    return run_stereo_chain_host({points, n_points_or_null, max_points, cloud_stride_points, T_host, P_host, norm_a, norm_b, left_bgr, right_bgr,
                                  bgr_pitch_bytes, bgr_frame_stride_bytes, depth_out, disp_out_or_null, rows, cols, n_frames, step, nc,
                                  iterations, use_superpixel, flags, params, stats_or_null},
                                 devices_or_null, n_devices, true);
}

int dcmt_measurement_derivatives_f32(const float* value, float* dx, float* dy, int rows, int cols, int n_frames,
                                     void* cuda_stream) {
    if (!value || !dx) return fail(DCMT_E_BADARG, "null pointer");
    int rc = check_planes(rows, cols, n_frames);
    if (rc) return rc;
    if ((rc = check_device())) return rc;
    API_CUDA(dcmt::stereo_measurement_derivatives(value, dx, dy, rows, cols, n_frames, static_cast<cudaStream_t>(cuda_stream)),
             "measurement derivatives launch");
    return DCMT_OK;
}

int dcmt_get_initial_disparity_f32(const float* depth, float* disp, int rows, int cols, int n_frames, float baseline,
                                   float focal, void* cuda_stream) {
    if (!depth || !disp) return fail(DCMT_E_BADARG, "null pointer");
    int rc = check_planes(rows, cols, n_frames);
    if (rc) return rc;
    if ((rc = check_device())) return rc;
    API_CUDA(dcmt::stereo_get_initial_disparity(depth, disp, rows, cols, n_frames, baseline, focal, static_cast<cudaStream_t>(cuda_stream)),
             "initial disparity launch");
    return DCMT_OK;
}

int dcmt_optimize_ig_f32(const float* value_left, const float* value_right, float* disp, int rows, int cols, int n_frames,
                         int num_iterations, float damp_factor, float err_clip, void* cuda_stream) {
    if (!value_left || !value_right || !disp) return fail(DCMT_E_BADARG, "null pointer");
    int rc = check_planes(rows, cols, n_frames);
    if (rc) return rc;
    if (num_iterations < 0) return fail(DCMT_E_BADARG, "num_iterations %d", num_iterations);
    if ((rc = check_device())) return rc;
    API_CUDA(dcmt::stereo_optimize_ig(value_left, value_right, disp, rows, cols, n_frames, num_iterations, damp_factor,
                                      err_clip, static_cast<cudaStream_t>(cuda_stream)),
             "optimize_IG launch");
    return DCMT_OK;
}

int dcmt_retrieve_optimized_depth_f32(const float* disp, float* depth, int rows, int cols, int n_frames, float baseline,
                                      float focal, float depth_clip, void* cuda_stream) {
    if (!disp || !depth) return fail(DCMT_E_BADARG, "null pointer");
    int rc = check_planes(rows, cols, n_frames);
    if (rc) return rc;
    if ((rc = check_device())) return rc;
    API_CUDA(dcmt::stereo_retrieve_depth(disp, depth, rows, cols, n_frames, baseline, focal, depth_clip, static_cast<cudaStream_t>(cuda_stream)),
             "retrieve depth launch");
    return DCMT_OK;
}

// ---- cv::cvtColor(COLOR_BGR2GRAY) in front of the EntryType fill (main_sl.cpp:1167,1171) ----
static int check_gray(const uint8_t* bgr, uint8_t* gray, int rows, int cols, size_t* bgr_pitch, size_t* gray_pitch, int n_frames) {
    if (!bgr || !gray) return fail(DCMT_E_BADARG, "null pointer");
    int rc = check_planes(rows, cols, n_frames);
    if (rc) return rc;
    if (rows > 65535 || n_frames > 65535) return fail(DCMT_E_UNSUPPORTED, "at most 65535 rows / frames");
    if (*bgr_pitch == 0) *bgr_pitch = (size_t)cols * 3;
    if (*gray_pitch == 0) *gray_pitch = (size_t)cols;
    if (*bgr_pitch < (size_t)cols * 3 || *gray_pitch < (size_t)cols) return fail(DCMT_E_BADARG, "pitch too small");
    return DCMT_OK;
}

int dcmt_bgr2gray_u8(const uint8_t* bgr, uint8_t* gray, int rows, int cols, size_t bgr_pitch_bytes, size_t gray_pitch_bytes, int n_frames,
                     void* cuda_stream) {
    int rc = check_gray(bgr, gray, rows, cols, &bgr_pitch_bytes, &gray_pitch_bytes, n_frames);
    if (rc) return rc;
    if (n_frames == 0) return DCMT_OK;
    if ((rc = check_device())) return rc;
    API_CUDA(dcmt::stereo_bgr2gray(bgr, bgr_pitch_bytes, bgr_pitch_bytes * rows, gray, gray_pitch_bytes, gray_pitch_bytes * rows, rows, cols,
                                   n_frames, static_cast<cudaStream_t>(cuda_stream)),
             "BGR2GRAY launch");
    return DCMT_OK;
}

int dcmt_bgr2gray_u8_host(const uint8_t* bgr, uint8_t* gray, int rows, int cols, size_t bgr_pitch_bytes, size_t gray_pitch_bytes, int n_frames) {
    int rc = check_gray(bgr, gray, rows, cols, &bgr_pitch_bytes, &gray_pitch_bytes, n_frames);
    if (rc) return rc;
    if (n_frames == 0) return DCMT_OK;
    const size_t in_row = (size_t)cols * 3, frames_rows = (size_t)rows * n_frames;
    Staged si{bgr, nullptr, bgr_pitch_bytes, in_row, frames_rows}, so{nullptr, gray, gray_pitch_bytes, (size_t)cols, frames_rows};
    return run_staged({&si, &so}, [&](cudaStream_t st) {
        return cuda_rc(dcmt::stereo_bgr2gray(static_cast<const uint8_t*>(si.dev), in_row, in_row * rows, static_cast<uint8_t*>(so.dev), cols,
                                             (size_t)cols * rows, rows, cols, n_frames, st), "BGR2GRAY launch");
    });
}

// ---- cv::cvtColor(COLOR_BGR2Lab) in front of Slic::generate_superpixels (main_lc.cpp:182-184, main_sl.cpp:438) ----
static int check_lab(const uint8_t* bgr, const uint8_t* lab, int rows, int cols, size_t* bgr_pitch, size_t* lab_pitch, int n_frames) {
    if (!bgr || !lab) return fail(DCMT_E_BADARG, "null pointer");
    int rc = check_planes(rows, cols, n_frames);
    if (rc) return rc;
    if (n_frames > 65535) return fail(DCMT_E_UNSUPPORTED, "at most 65535 frames");
    if ((size_t)rows * (size_t)cols >= (size_t)1 << 31) return fail(DCMT_E_UNSUPPORTED, "frame of 2^31 pixels or more");
    const size_t row = (size_t)cols * 3;
    if (*bgr_pitch == 0) *bgr_pitch = row;
    if (*lab_pitch == 0) *lab_pitch = row;
    if (*bgr_pitch < row || *lab_pitch < row) return fail(DCMT_E_BADARG, "pitch too small");
    if (n_frames == 0) return DCMT_OK;
    // the byte ranges the call reads and writes must not overlap (no aliasing, dcmt.h)
    const size_t last = (size_t)rows * n_frames - 1;
    const uintptr_t in = reinterpret_cast<uintptr_t>(bgr), out = reinterpret_cast<uintptr_t>(lab);
    if (in < out + *lab_pitch * last + row && out < in + *bgr_pitch * last + row) return fail(DCMT_E_BADARG, "input and output overlap");
    return DCMT_OK;
}

int dcmt_bgr2lab_u8(const uint8_t* bgr, uint8_t* lab, int rows, int cols, size_t bgr_pitch_bytes, size_t lab_pitch_bytes, int n_frames,
                    void* cuda_stream) {
    int rc = check_lab(bgr, lab, rows, cols, &bgr_pitch_bytes, &lab_pitch_bytes, n_frames);
    if (rc) return rc;
    if (n_frames == 0) return DCMT_OK;
    if ((rc = check_device())) return rc;
    API_CUDA(dcmt::color_bgr2lab(bgr, bgr_pitch_bytes, bgr_pitch_bytes * rows, lab, lab_pitch_bytes, lab_pitch_bytes * rows, rows, cols,
                                 n_frames, static_cast<cudaStream_t>(cuda_stream)),
             "BGR2Lab launch");
    return DCMT_OK;
}

int dcmt_bgr2lab_u8_host(const uint8_t* bgr, uint8_t* lab, int rows, int cols, size_t bgr_pitch_bytes, size_t lab_pitch_bytes, int n_frames) {
    int rc = check_lab(bgr, lab, rows, cols, &bgr_pitch_bytes, &lab_pitch_bytes, n_frames);
    if (rc) return rc;
    if (n_frames == 0) return DCMT_OK;
    const size_t row = (size_t)cols * 3, frames_rows = (size_t)rows * n_frames;
    Staged si{bgr, nullptr, bgr_pitch_bytes, row, frames_rows}, so{nullptr, lab, lab_pitch_bytes, row, frames_rows};
    return run_staged({&si, &so}, [&](cudaStream_t st) {
        return cuda_rc(dcmt::color_bgr2lab(static_cast<const uint8_t*>(si.dev), row, row * rows, static_cast<uint8_t*>(so.dev), row, row * rows,
                                           rows, cols, n_frames, st), "BGR2Lab launch");
    });
}

// ---- (a3) the reference's own containers: EntryType matrices and pitched CV_32FC1 matrices with in-place semantics ----
static int check_entries(const void* e, int rows, int cols, size_t row_step, size_t elem_stride) {
    if (!e) return fail(DCMT_E_BADARG, "null pointer");
    int rc = check_planes(rows, cols, 1);
    if (rc) return rc;
    if (rows > 65535) return fail(DCMT_E_UNSUPPORTED, "at most 65535 rows");
    if (elem_stride < 12 || elem_stride % 4 != 0) return fail(DCMT_E_BADARG, "elem_stride_bytes %zu: EntryType is three floats", elem_stride);
    if (row_step % 4 != 0 || row_step < (size_t)cols * elem_stride) return fail(DCMT_E_BADARG, "row_step_bytes %zu invalid for %d entries of %zu bytes", row_step, cols, elem_stride);
    if (reinterpret_cast<uintptr_t>(e) % 4 != 0) return fail(DCMT_E_BADARG, "entries must be 4-byte aligned");
    return DCMT_OK;
}
static int check_mat_f32(const float* p, int rows, int cols, size_t* pitch_bytes) {
    if (!p) return fail(DCMT_E_BADARG, "null pointer");
    if (*pitch_bytes == 0) *pitch_bytes = (size_t)cols * sizeof(float);
    if (*pitch_bytes % sizeof(float) != 0 || *pitch_bytes < (size_t)cols * sizeof(float)) return fail(DCMT_E_BADARG, "pitch_bytes %zu invalid", *pitch_bytes);
    return DCMT_OK;
}

int dcmt_entries_measurement_derivatives(void* entries, int rows, int cols, size_t row_step_bytes, size_t elem_stride_bytes, void* cuda_stream) {
    int rc = check_entries(entries, rows, cols, row_step_bytes, elem_stride_bytes);
    if (rc) return rc;
    if ((rc = check_device())) return rc;
    API_CUDA(dcmt::stereo_entries_derivatives(entries, row_step_bytes, elem_stride_bytes, rows, cols, static_cast<cudaStream_t>(cuda_stream)),
             "measurement derivatives launch");
    return DCMT_OK;
}

static int check_entries_optimize_ig(const void* entries_left, size_t left_row_step_bytes, const void* entries_right,
                                     size_t right_row_step_bytes, size_t elem_stride_bytes, const float* disp, size_t* disp_pitch_bytes,
                                     int rows, int cols, int num_iterations) {
    int rc = check_entries(entries_left, rows, cols, left_row_step_bytes, elem_stride_bytes);
    if (rc) return rc;
    if ((rc = check_entries(entries_right, rows, cols, right_row_step_bytes, elem_stride_bytes))) return rc;
    if ((rc = check_mat_f32(disp, rows, cols, disp_pitch_bytes))) return rc;
    if (num_iterations < 0) return fail(DCMT_E_BADARG, "num_iterations %d", num_iterations);
    return DCMT_OK;
}

int dcmt_entries_optimize_ig(const void* entries_left, size_t left_row_step_bytes, const void* entries_right, size_t right_row_step_bytes,
                             size_t elem_stride_bytes, float* disp, size_t disp_pitch_bytes, int rows, int cols, int num_iterations,
                             float damp_factor, float err_clip, void* cuda_stream) {
    int rc = check_entries_optimize_ig(entries_left, left_row_step_bytes, entries_right, right_row_step_bytes, elem_stride_bytes, disp,
                                       &disp_pitch_bytes, rows, cols, num_iterations);
    if (rc) return rc;
    if ((rc = check_device())) return rc;
    API_CUDA(dcmt::stereo_entries_optimize_ig(entries_left, left_row_step_bytes, entries_right, right_row_step_bytes, elem_stride_bytes, disp,
                                              disp_pitch_bytes / sizeof(float), rows, cols, num_iterations, damp_factor, err_clip,
                                              static_cast<cudaStream_t>(cuda_stream)),
             "optimize_IG launch");
    return DCMT_OK;
}

// the two CV_32FC1 Mat operations, input then output
static int check_mat_pair(const float* in, size_t* in_pitch_bytes, const float* out, size_t* out_pitch_bytes, int rows, int cols) {
    int rc = check_planes(rows, cols, 1);
    if (rc) return rc;
    if (rows > 65535) return fail(DCMT_E_UNSUPPORTED, "at most 65535 rows");
    if ((rc = check_mat_f32(in, rows, cols, in_pitch_bytes)) || (rc = check_mat_f32(out, rows, cols, out_pitch_bytes))) return rc;
    return DCMT_OK;
}

int dcmt_get_initial_disparity_mat_f32(const float* depth, size_t depth_pitch_bytes, float* disp, size_t disp_pitch_bytes, int rows, int cols,
                                       float baseline, float focal, void* cuda_stream) {
    int rc = check_mat_pair(depth, &depth_pitch_bytes, disp, &disp_pitch_bytes, rows, cols);
    if (rc) return rc;
    if ((rc = check_device())) return rc;
    API_CUDA(dcmt::stereo_initial_disparity_mat(depth, depth_pitch_bytes / sizeof(float), disp, disp_pitch_bytes / sizeof(float), rows, cols,
                                                baseline, focal, static_cast<cudaStream_t>(cuda_stream)),
             "initial disparity launch");
    return DCMT_OK;
}

int dcmt_retrieve_optimized_depth_mat_f32(const float* disp, size_t disp_pitch_bytes, float* depth, size_t depth_pitch_bytes, int rows, int cols,
                                          float baseline, float focal, float depth_clip, void* cuda_stream) {
    int rc = check_mat_pair(disp, &disp_pitch_bytes, depth, &depth_pitch_bytes, rows, cols);
    if (rc) return rc;
    if ((rc = check_device())) return rc;
    API_CUDA(dcmt::stereo_retrieve_depth_mat(disp, disp_pitch_bytes / sizeof(float), depth, depth_pitch_bytes / sizeof(float), rows, cols,
                                             baseline, focal, depth_clip, static_cast<cudaStream_t>(cuda_stream)),
             "retrieve depth launch");
    return DCMT_OK;
}

// host variants: the used part of every row goes to the device (cols * elem_stride bytes of a row_step-byte row), the
// kernels run on the packed copy, and what the reference function modifies comes back
int dcmt_entries_measurement_derivatives_host(void* entries, int rows, int cols, size_t row_step_bytes, size_t elem_stride_bytes) {
    int rc = check_entries(entries, rows, cols, row_step_bytes, elem_stride_bytes);
    if (rc) return rc;
    const size_t used = (size_t)cols * elem_stride_bytes;
    Staged se{entries, entries, row_step_bytes, used, (size_t)rows};
    return run_staged({&se}, [&](cudaStream_t st) {
        return cuda_rc(dcmt::stereo_entries_derivatives(se.dev, used, elem_stride_bytes, rows, cols, st), "measurement derivatives launch");
    });
}

int dcmt_entries_optimize_ig_host(const void* entries_left, size_t left_row_step_bytes, const void* entries_right,
                                  size_t right_row_step_bytes, size_t elem_stride_bytes, float* disp, size_t disp_pitch_bytes, int rows,
                                  int cols, int num_iterations, float damp_factor, float err_clip) {
    int rc = check_entries_optimize_ig(entries_left, left_row_step_bytes, entries_right, right_row_step_bytes, elem_stride_bytes, disp,
                                       &disp_pitch_bytes, rows, cols, num_iterations);
    if (rc) return rc;
    const size_t used = (size_t)cols * elem_stride_bytes;
    Staged sl{entries_left, nullptr, left_row_step_bytes, used, (size_t)rows}, sr{entries_right, nullptr, right_row_step_bytes, used, (size_t)rows},
        sd{disp, disp, disp_pitch_bytes, (size_t)cols * sizeof(float), (size_t)rows};
    return run_staged({&sl, &sr, &sd}, [&](cudaStream_t st) {
        return cuda_rc(dcmt::stereo_entries_optimize_ig(sl.dev, used, sr.dev, used, elem_stride_bytes, static_cast<float*>(sd.dev), cols, rows, cols,
                                                        num_iterations, damp_factor, err_clip, st), "optimize_IG launch");
    });
}

// the output is copied in as well: pixels the kernel skips keep the caller's value
int dcmt_get_initial_disparity_mat_f32_host(const float* depth, size_t depth_pitch_bytes, float* disp, size_t disp_pitch_bytes, int rows,
                                            int cols, float baseline, float focal) {
    int rc = check_mat_pair(depth, &depth_pitch_bytes, disp, &disp_pitch_bytes, rows, cols);
    if (rc) return rc;
    const size_t row = (size_t)cols * sizeof(float);
    Staged si{depth, nullptr, depth_pitch_bytes, row, (size_t)rows}, so{disp, disp, disp_pitch_bytes, row, (size_t)rows};
    return run_staged({&si, &so}, [&](cudaStream_t st) {
        return cuda_rc(dcmt::stereo_initial_disparity_mat(static_cast<const float*>(si.dev), cols, static_cast<float*>(so.dev), cols, rows, cols,
                                                          baseline, focal, st), "initial disparity launch");
    });
}

int dcmt_retrieve_optimized_depth_mat_f32_host(const float* disp, size_t disp_pitch_bytes, float* depth, size_t depth_pitch_bytes, int rows,
                                               int cols, float baseline, float focal, float depth_clip) {
    int rc = check_mat_pair(disp, &disp_pitch_bytes, depth, &depth_pitch_bytes, rows, cols);
    if (rc) return rc;
    const size_t row = (size_t)cols * sizeof(float);
    Staged si{disp, nullptr, disp_pitch_bytes, row, (size_t)rows}, so{depth, depth, depth_pitch_bytes, row, (size_t)rows};
    return run_staged({&si, &so}, [&](cudaStream_t st) {
        return cuda_rc(dcmt::stereo_retrieve_depth_mat(static_cast<const float*>(si.dev), cols, static_cast<float*>(so.dev), cols, rows, cols,
                                                       baseline, focal, depth_clip, st), "retrieve depth launch");
    });
}

}  // extern "C"
