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
// must not be used); every caller checks arena_ok() before launching.
template <class T>
T* carve(Arena* a, size_t count) {
    const size_t bytes = (count * sizeof(T) + 255) & ~size_t(255);
    if (a->used + bytes > a->cap) {
        a->overflow = true;
        return reinterpret_cast<T*>(a->base);
    }
    T* p = reinterpret_cast<T*>(a->base + a->used);
    a->used += bytes;
    return p;
}
int arena_ok(const Arena* a) {
    return a->overflow ? fail(DCMT_E_NOMEM, "internal: workspace arena of %zu bytes is too small for this call", a->cap) : DCMT_OK;
}
size_t carve_bytes(size_t count, size_t elem) { return (count * elem + 255) & ~size_t(255); }

// frames per generic chunk: a 2^27-pixel budget split evenly (313 KITTI frames, 1 GB of float scratch).  Larger grids
// beat L2 residency of the two float planes here as well (20-frame chunks were 10 % slower).
int generic_chunk_frames(int rows, int cols, int n_frames) {
    static const long env = [] {
        const char* s = getenv("DCMT_GENERIC_CHUNK");
        return s ? atol(s) : 0L;
    }();
    long cap = env > 0 ? env : (long)(((size_t)1 << 27) / ((size_t)rows * cols));
    if (cap < 1) cap = 1;
    if (cap > 65535) cap = 65535;
    const long nchunks = (n_frames + cap - 1) / cap;
    long c = nchunks > 0 ? (n_frames + nchunks - 1) / nchunks : 1;
    if (c < 1) c = 1;
    return (int)c;
}

// frames per fused chunk: as many as a 2^28-pixel budget allows (627 KITTI frames; about 0.5 GB of uint16 intermediate
// plus 2 GB of fix-up scratch), split evenly.  Large grids matter more than L2 residency of the intermediate plane:
// the kernels are issue-bound (DRAM a few per cent busy), while every launch ends in a partially filled wave
// (79-frame chunks: 8.5 waves per launch, 11 % slower end to end than 512-frame chunks on the B200).
int fused_chunk_frames(int rows, int cols, int n_frames) {
    static const long env = [] {
        const char* s = getenv("DCMT_FUSED_CHUNK");
        return s ? atol(s) : 0L;
    }();
    long cap = env > 0 ? env : (long)(((size_t)1 << 28) / ((size_t)rows * cols));
    if (cap < 1) cap = 1;
    if (cap > 65535) cap = 65535;
    const long nchunks = (n_frames + cap - 1) / cap;
    long c = nchunks > 0 ? (n_frames + nchunks - 1) / nchunks : 1;
    if (c < 1) c = 1;
    return (int)c;
}

size_t generic_ws_bytes(int rows, int cols, int chunk, bool bilateral) {
    const size_t fpix = (size_t)rows * cols;
    size_t b = 2 * carve_bytes(fpix * chunk, sizeof(float)) + carve_bytes(chunk, sizeof(dcmt::FrameCounters));
    if (bilateral) b += carve_bytes(2 * (size_t)chunk, sizeof(unsigned)) + carve_bytes(dcmt::generic_lut_floats() * chunk, sizeof(float));
    return b;
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

int check_geometry(int rows, int cols, size_t pitch_bytes, size_t frame_stride_bytes, int n_frames, Geometry* g,
                   size_t elem = sizeof(float)) {
    if (rows < 1 || cols < 1) return fail(DCMT_E_BADARG, "rows and cols must be >= 1 (got %d x %d)", rows, cols);
    if (n_frames < 0) return fail(DCMT_E_BADARG, "n_frames must be >= 0 (got %d)", n_frames);
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

// validated description of one completion call
struct CompletionCall {
    const int32_t* labels;
    int n_clusters;
    bool guided;
    int rows, cols, blur, flags;
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

size_t completion_ws_bytes(int rows, int cols, int n_frames, bool bilateral, bool fused, bool u16_in = false, bool rank = false) {
    const int chunk = fused ? fused_chunk_frames(rows, cols, n_frames) : generic_chunk_frames(rows, cols, n_frames);
    size_t b = generic_ws_bytes(rows, cols, chunk, bilateral);
    if (fused && rank) {  // dictionary, its sizes, the code plane (rank_f32.cu)
        const size_t code_pitch = ((size_t)cols + 7) / 8 * 8;
        b += carve_bytes((size_t)dcmt::kRankMaxValid * chunk, sizeof(float)) + carve_bytes((size_t)chunk, sizeof(int)) +
             carve_bytes((size_t)rows * code_pitch * chunk, sizeof(uint16_t));
    }
    if (u16_in && !fused) b += carve_bytes((size_t)rows * cols * chunk, sizeof(float));
    if (fused) {
        const size_t mid_pitch = ((size_t)cols + 7) / 8 * 8;
        b += carve_bytes((size_t)rows * mid_pitch * chunk, sizeof(uint16_t)) + 2 * carve_bytes(mid_pitch * chunk, sizeof(uint32_t));
        b += carve_bytes(((size_t)rows / 8 + 1) * ((size_t)cols / 8 + 1) * chunk, sizeof(int));  // tile flags of the guided front (upper bound)
    }
    return b;
}

// Enqueue n_frames through the pipeline; every pointer is a device pointer, the workspace is carved from `ar`.
// Never synchronises.  On the fused path `redo_flags` (device, one int32 per frame, optional) receives 1 for
// frames that turned out not to be strict q8: their output is NOT valid and the caller must redo them with
// DCMT_PATH_GENERIC.  *used_fused tells the caller which path ran.
//
// Input is either float32 metres (`sparse`, sharing pitch / fstride with the output) or -- `in16.p` non-null -- KITTI
// uint16 (metres * 256, main.cpp:75-82) with its own pitch / frame stride in elements.  uint16 input is strict q8 by
// construction: the fused kernels read it directly and nothing is validated or redone; shapes the fused kernels do
// not serve get a convertTo(CV_32F, 1/256) (main.cpp:79) into a workspace plane in front of the generic pipeline.
struct U16Input {
    const uint16_t* p = nullptr;
    size_t pitch = 0, fstride = 0;  // elements
};

int enqueue_completion(const CompletionCall& cc, const float* sparse, const int32_t* labels, float* dense, size_t pitch,
                       size_t fstride, int n_frames, int32_t* stats, int32_t* redo_flags, float* stages,
                       uint32_t* stage_mask, Arena* ar, cudaStream_t st, bool* used_fused, U16Input in16 = U16Input{}) {
    const int rows = cc.rows, cols = cc.cols;
    const bool bilateral = cc.blur == DCMT_BLUR_BILATERAL;
    const bool fused = fused_applies(cc) && !stages;
    const int chunk = fused ? fused_chunk_frames(rows, cols, n_frames) : generic_chunk_frames(rows, cols, n_frames);
    if (used_fused) *used_fused = fused;
    const size_t fpix = (size_t)rows * cols;
    float* w1 = carve<float>(ar, fpix * chunk);
    float* w2 = carve<float>(ar, fpix * chunk);
    dcmt::FrameCounters* ctr = carve<dcmt::FrameCounters>(ar, chunk);
    unsigned* mm = bilateral ? carve<unsigned>(ar, 2 * (size_t)chunk) : nullptr;
    float* lut = bilateral ? carve<float>(ar, dcmt::generic_lut_floats() * chunk) : nullptr;
    if (fused) {
        dcmt::Q8Plan p{};
        p.rows = rows;
        p.cols = cols;
        dcmt::q8_choose_tile(rows, cols, &p.th, &p.tw);
        p.mid_pitch = (cols + 7) / 8 * 8;
        p.max_frames = chunk;
        p.mid = carve<uint16_t>(ar, (size_t)rows * p.mid_pitch * chunk);
        p.col_first = carve<uint32_t>(ar, (size_t)p.mid_pitch * chunk);
        p.col_last = carve<uint32_t>(ar, (size_t)p.mid_pitch * chunk);
        p.ctr = ctr;
        p.w1 = w1;
        p.w2 = w2;
        int* tile_flags = cc.guided ? carve<int>(ar, dcmt::q8_guided_tile_flags(rows, cols, p.th, p.tw, chunk)) : nullptr;
        // DCMT_PATH_RANK: float32 frames through the per-frame dictionary (rank_f32.cu) in front of the same kernels
        const bool rank = cc.flags == DCMT_PATH_RANK && !in16.p;
        float* lut = rank ? carve<float>(ar, (size_t)dcmt::kRankMaxValid * chunk) : nullptr;
        int* lut_count = rank ? carve<int>(ar, (size_t)chunk) : nullptr;
        uint16_t* codes = rank ? carve<uint16_t>(ar, (size_t)rows * p.mid_pitch * chunk) : nullptr;
        if (int rc = arena_ok(ar)) return rc;
        if (rank) {
            API_CUDA(dcmt::rank_configure(), "kernel attribute setup");
            p.codes_in = 1;
            p.counters_ready = 1;
            p.lut = lut;
        }
        for (int f0 = 0; f0 < n_frames; f0 += chunk) {
            const int nf = n_frames - f0 < chunk ? n_frames - f0 : chunk;
            ProfEvents pe{};
            API_CUDA(prof_mark(st, 0, &pe), "profiling event");
            if (rank) {
                API_CUDA(dcmt::q8_zero_counters(p, nf, st), "counter setup launch");
                API_CUDA(dcmt::rank_build(sparse + (size_t)f0 * fstride, pitch, fstride, rows, cols, nf, lut, lut_count, codes,
                                          (size_t)p.mid_pitch, ctr, st),
                         "dictionary launch");
                if (cc.guided)
                    API_CUDA(dcmt::q8_run_guided_front(p, nullptr, codes, (size_t)p.mid_pitch, (size_t)p.mid_pitch * rows,
                                                       labels + (size_t)f0 * fpix, cc.n_clusters, nf, 0, tile_flags, st),
                             "fused guided front launch");
                else
                    API_CUDA(dcmt::q8_run_front(p, nullptr, codes, (size_t)p.mid_pitch, (size_t)p.mid_pitch * rows, nf, 0, st),
                             "fused front launch");
            } else if (cc.guided)
                API_CUDA(dcmt::q8_run_guided_front(p, sparse + (size_t)f0 * fstride, nullptr, pitch, fstride, labels + (size_t)f0 * fpix,
                                                   cc.n_clusters, nf, cc.flags != DCMT_PATH_FUSED, tile_flags, st),
                         "fused guided front launch");
            else if (in16.p)
                API_CUDA(dcmt::q8_run_front(p, nullptr, in16.p + (size_t)f0 * in16.fstride, in16.pitch, in16.fstride, nf, 0, st),
                         "fused front launch");
            else
                API_CUDA(dcmt::q8_run_front(p, sparse + (size_t)f0 * fstride, nullptr, pitch, fstride, nf,
                                            cc.flags != DCMT_PATH_FUSED, st),
                         "fused front launch");
            API_CUDA(prof_mark(st, 1, &pe), "profiling event");
            API_CUDA(dcmt::q8_run_tail(p, dense + (size_t)f0 * fstride, pitch, fstride, nf, cc.blur, st), "fused tail launch");
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
    float* conv = in16.p ? carve<float>(ar, fpix * chunk) : nullptr;
    if (int rc = arena_ok(ar)) return rc;
    for (int f0 = 0; f0 < n_frames; f0 += chunk) {
        const int nf = n_frames - f0 < chunk ? n_frames - f0 : chunk;
        dcmt::GenericChunk c{};
        if (in16.p) {
            API_CUDA(dcmt::q8_convert_u16(in16.p + (size_t)f0 * in16.fstride, in16.pitch, in16.fstride, conv, rows, cols, nf, st),
                     "uint16 conversion launch");
            c.in = conv;
            c.in_pitch = (size_t)cols;
            c.in_fstride = fpix;
        } else {
            c.in = sparse + (size_t)f0 * fstride;
            c.in_pitch = pitch;
            c.in_fstride = fstride;
        }
        c.labels = cc.guided ? labels + (size_t)f0 * fpix : nullptr;
        c.n_clusters = cc.n_clusters;
        c.guided = cc.guided;
        c.out = dense + (size_t)f0 * fstride;
        c.out_pitch = pitch;
        c.out_fstride = fstride;
        c.rows = rows;
        c.cols = cols;
        c.n_frames = nf;
        c.blur = cc.blur;
        c.w1 = w1;
        c.w2 = w2;
        c.ctr = ctr;
        c.minmax = mm;
        c.lut = lut;
        c.stats = stats ? stats + (size_t)f0 * DCMT_STATS_STRIDE : nullptr;
        c.stages = stages;
        c.stage_mask = stage_mask;
        c.skip_front = false;
        API_CUDA(dcmt::generic_run_chunk(c, st), "generic pipeline launch");
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

int validate_completion(const float* sparse, const int32_t* labels, bool guided, float* dense, int rows, int cols,
                        size_t pitch_bytes, size_t frame_stride_bytes, int n_frames, int blur_type, int flags, Geometry* g) {
    if (!sparse || !dense) return fail(DCMT_E_BADARG, "null image pointer");
    if (guided && !labels) return fail(DCMT_E_BADARG, "null label pointer");
    if (blur_type < DCMT_BLUR_NONE || blur_type > DCMT_BLUR_BILATERAL) return fail(DCMT_E_BADARG, "blur_type %d", blur_type);
    if (flags < DCMT_PATH_AUTO || flags > DCMT_PATH_RANK) return fail(DCMT_E_BADARG, "flags %d", flags);
    int rc = check_geometry(rows, cols, pitch_bytes, frame_stride_bytes, n_frames, g);
    if (rc) return rc;
    if (n_frames && overlaps(sparse, g->span_bytes, dense, g->span_bytes)) return fail(DCMT_E_BADARG, "input and output overlap");
    return DCMT_OK;
}

// device-pointer driver of (a1) and (a2)
int run_completion(const float* sparse, const int32_t* labels, int n_clusters, bool guided, float* dense, int rows,
                   int cols, size_t pitch_bytes, size_t frame_stride_bytes, int n_frames, int blur_type, int flags,
                   int32_t* stats, float* stages, uint32_t* stage_mask, cudaStream_t st) {
    Geometry g;
    int rc = validate_completion(sparse, labels, guided, dense, rows, cols, pitch_bytes, frame_stride_bytes, n_frames,
                                 blur_type, flags, &g);
    if (rc) return rc;
    if (n_frames == 0) return DCMT_OK;
    if ((rc = check_device())) return rc;
    API_CUDA(dcmt::generic_configure(), "kernel attribute setup");
    API_CUDA(dcmt::q8_configure(), "kernel attribute setup");
    CompletionCall cc{labels, n_clusters, guided, rows, cols, blur_type, flags};
    const bool fused = fused_applies(cc) && !stages;
    const bool bilateral = blur_type == DCMT_BLUR_BILATERAL;
    Arena* ar = nullptr;
    const size_t flag_bytes = fused ? carve_bytes((size_t)n_frames, sizeof(int32_t)) : 0;
    if ((rc = arena_acquire(st, completion_ws_bytes(rows, cols, n_frames, bilateral, fused, false, flags == DCMT_PATH_RANK) + flag_bytes, &ar)))
        return rc;
    int32_t* d_flags = fused ? carve<int32_t>(ar, (size_t)n_frames) : nullptr;
    bool used = false;
    if ((rc = enqueue_completion(cc, sparse, labels, dense, g.pitch, g.fstride, n_frames, stats, d_flags, stages, stage_mask, ar,
                                 st, &used)))
        return rc;
    if (!used || flags == DCMT_PATH_FUSED || flags == DCMT_PATH_GENERIC) return DCMT_OK;  // DCMT_PATH_FUSED: fully asynchronous, stats[3] = -1 marks bad frames
    // DCMT_PATH_AUTO / DCMT_PATH_RANK: read the per-frame "not served" flags back (one synchronisation per pass) and redo
    // those frames one level down: strict-q8 kernels -> dictionary (rank_f32.cu) -> generic pipeline
    int32_t* h_flags = nullptr;
    if ((rc = pinned_flags(st, (size_t)n_frames, &h_flags))) return rc;
    API_CUDA(cudaMemcpyAsync(h_flags, d_flags, (size_t)n_frames * sizeof(int32_t), cudaMemcpyDeviceToHost, st), "flag readback");
    API_CUDA(cudaStreamSynchronize(st), "kernel execution");
    for (int level = flags == DCMT_PATH_AUTO ? DCMT_PATH_RANK : DCMT_PATH_GENERIC;; level = DCMT_PATH_GENERIC) {
        cc.flags = level;
        const bool want_flags = level == DCMT_PATH_RANK;
        bool any = false;
        for (int f = 0; f < n_frames;) {
            if (!h_flags[f]) { ++f; continue; }
            int e = f;
            while (e < n_frames && h_flags[e]) ++e;
            // the previous pass has completed (stream synchronised): the arena is free again, but it was sized for that
            // pass -- this one may need more (the generic pipeline: two float planes per frame of its chunk)
            const size_t fb = want_flags ? carve_bytes((size_t)(e - f), sizeof(int32_t)) : 0;
            if ((rc = arena_acquire(st, completion_ws_bytes(rows, cols, e - f, bilateral, want_flags, false, want_flags) + fb, &ar))) return rc;
            int32_t* run_flags = want_flags ? carve<int32_t>(ar, (size_t)(e - f)) : nullptr;
            if ((rc = enqueue_completion(cc, sparse + (size_t)f * g.fstride, guided ? labels + (size_t)f * rows * cols : nullptr,
                                         dense + (size_t)f * g.fstride, g.pitch, g.fstride, e - f,
                                         stats ? stats + (size_t)f * DCMT_STATS_STRIDE : nullptr, run_flags, nullptr, nullptr, ar, st, nullptr)))
                return rc;
            if (want_flags) {
                // arenas are reused by the next run of this pass in stream order; the flags leave through the pinned buffer first
                API_CUDA(cudaMemcpyAsync(h_flags + f, run_flags, (size_t)(e - f) * sizeof(int32_t), cudaMemcpyDeviceToHost, st), "flag readback");
                API_CUDA(cudaStreamSynchronize(st), "kernel execution");
            }
            any = true;
            f = e;
        }
        if (level == DCMT_PATH_GENERIC || !any) break;
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

int copy_frames_d2h(void* h, size_t h_pitch_bytes, size_t h_fstride_bytes, const void* d, size_t row_bytes, int rows, int nf, cudaStream_t st) {
    if (h_pitch_bytes == row_bytes && h_fstride_bytes == row_bytes * rows) {
        API_CUDA(cudaMemcpyAsync(h, d, row_bytes * rows * nf, cudaMemcpyDeviceToHost, st), "device to host copy");
    } else if (h_fstride_bytes == h_pitch_bytes * (size_t)rows) {
        API_CUDA(cudaMemcpy2DAsync(h, h_pitch_bytes, d, row_bytes, row_bytes, (size_t)rows * nf, cudaMemcpyDeviceToHost, st), "device to host copy");
    } else {
        for (int f = 0; f < nf; ++f)
            API_CUDA(cudaMemcpy2DAsync(static_cast<char*>(h) + (size_t)f * h_fstride_bytes, h_pitch_bytes,
                                       static_cast<const char*>(d) + (size_t)f * rows * row_bytes, row_bytes, row_bytes, rows,
                                       cudaMemcpyDeviceToHost, st),
                     "device to host copy");
    }
    return DCMT_OK;
}

// copy_only: the same buffers, chunking and streams with the kernels left out (the input is echoed to the output) --
// the ceiling the host <-> device links put on the end-to-end rate (dcmt_debug_host_copy_*).
int run_completion_host(const float* sparse, const int32_t* labels, int n_clusters, bool guided, float* dense, int rows,
                        int cols, size_t pitch_bytes, size_t frame_stride_bytes, int n_frames, int blur_type, int flags,
                        int32_t* stats, const int* devices = nullptr, int n_devices = 0, bool multi = false, bool copy_only = false) {
    Geometry g;
    int rc = validate_completion(sparse, labels, guided, dense, rows, cols, pitch_bytes, frame_stride_bytes, n_frames,
                                 blur_type, flags, &g);
    if (rc) return rc;
    if (n_frames == 0) return DCMT_OK;
    HostCall call;
    if ((rc = call.open(devices, n_devices, multi))) return rc;
    call.split(n_frames);
    const size_t fpix = (size_t)rows * cols;
    const bool bilateral = blur_type == DCMT_BLUR_BILATERAL;
    const size_t row_bytes = (size_t)cols * sizeof(float);
    const CompletionCall cc{labels, n_clusters, guided, rows, cols, blur_type, flags};
    const bool fused = fused_applies(cc) && !copy_only;
    int longest = 0;
    for (Lane& l : call.lanes) longest = std::max(longest, l.f_end - l.f_begin);
    const int hc = host_chunk_frames(rows, cols, longest);
    const size_t bytes = 2 * carve_bytes(fpix * hc, sizeof(float)) + (guided ? carve_bytes(fpix * hc, sizeof(int32_t)) : 0) +
                         carve_bytes((size_t)hc * DCMT_STATS_STRIDE, sizeof(int32_t)) + carve_bytes((size_t)hc, sizeof(int32_t)) +
                         completion_ws_bytes(rows, cols, hc, bilateral, fused, false, flags == DCMT_PATH_RANK);
    for (Lane& l : call.lanes) {
        if (l.f_end == l.f_begin) continue;
        if ((rc = call.use(l))) return rc;
        API_CUDA(dcmt::generic_configure(), "kernel attribute setup");
        API_CUDA(dcmt::q8_configure(), "kernel attribute setup");
        if (fused && (rc = pinned_flags(nullptr, (size_t)(l.f_end - l.f_begin), &l.h_flags))) return rc;
    }
    // one chunk [f0, f0 + nf) of lane l on its next stream: H2D, kernels, D2H
    auto do_chunk = [&](Lane& l, int f0, int nf, const CompletionCall& c2, bool fused2, int hc2, size_t bytes2) -> int {
        int rc2;
        cudaStream_t st = l.hs->s[l.slot];
        l.slot = (l.slot + 1) % kHostStreams;
        Arena* ar = nullptr;
        if ((rc2 = arena_acquire(st, bytes2, &ar))) return rc2;  // stream order protects reuse by the chunk 3 steps later
        float* d_in = carve<float>(ar, fpix * hc2);
        float* d_out = carve<float>(ar, fpix * hc2);
        int32_t* d_lab = guided ? carve<int32_t>(ar, fpix * hc2) : nullptr;
        int32_t* d_stats = carve<int32_t>(ar, (size_t)hc2 * DCMT_STATS_STRIDE);
        int32_t* d_flags = carve<int32_t>(ar, (size_t)hc2);
        if ((rc2 = arena_ok(ar))) return rc2;
        if ((rc2 = copy_frames_h2d(d_in, row_bytes, sparse + (size_t)f0 * g.fstride, g.pitch * sizeof(float), g.fstride * sizeof(float),
                                   row_bytes, rows, nf, st)))
            return rc2;
        if (guided)
            API_CUDA(cudaMemcpyAsync(d_lab, labels + (size_t)f0 * fpix, fpix * nf * sizeof(int32_t), cudaMemcpyHostToDevice, st),
                     "host to device copy");
        if (copy_only) {
            d_out = d_in;
        } else if ((rc2 = enqueue_completion(c2, d_in, d_lab, d_out, cols, fpix, nf, stats ? d_stats : nullptr, fused2 ? d_flags : nullptr,
                                             nullptr, nullptr, ar, st, nullptr))) {
            return rc2;
        }
        if (fused2)
            API_CUDA(cudaMemcpyAsync(l.h_flags + (f0 - l.f_begin), d_flags, (size_t)nf * sizeof(int32_t), cudaMemcpyDeviceToHost, st),
                     "flag readback");
        if ((rc2 = copy_frames_d2h(dense + (size_t)f0 * g.fstride, g.pitch * sizeof(float), g.fstride * sizeof(float), d_out, row_bytes, rows,
                                   nf, st)))
            return rc2;
        if (stats && !copy_only)
            API_CUDA(cudaMemcpyAsync(stats + (size_t)f0 * DCMT_STATS_STRIDE, d_stats, (size_t)nf * DCMT_STATS_STRIDE * sizeof(int32_t),
                                     cudaMemcpyDeviceToHost, st),
                     "device to host copy");
        return DCMT_OK;
    };
    for (bool more = true; more;) {
        more = false;
        for (Lane& l : call.lanes) {
            if (l.next >= l.f_end) continue;
            more = true;
            if ((rc = call.use(l))) return rc;
            const int f0 = l.next, nf = std::min(hc, l.f_end - f0);
            l.next += nf;
            if ((rc = do_chunk(l, f0, nf, cc, fused, hc, bytes))) return rc;
        }
    }
    if ((rc = call.finish())) return rc;
    if (fused && (flags == DCMT_PATH_AUTO || flags == DCMT_PATH_RANK)) {
        // frames the pass did not serve (not strict q8; dictionary too small) are redone one level down -- strict-q8
        // kernels -> dictionary (rank_f32.cu) -> generic pipeline -- in runs of consecutive frames, on the device that
        // served them, through the same chunk pipeline
        for (int level = flags == DCMT_PATH_AUTO ? DCMT_PATH_RANK : DCMT_PATH_GENERIC;; level = DCMT_PATH_GENERIC) {
            CompletionCall cg = cc;
            cg.flags = level;
            const bool lf = level == DCMT_PATH_RANK;
            bool any = false;
            // the runs are fixed before anything is enqueued: the rank pass overwrites the flags it reads
            struct Run { Lane* l; int f, e; };
            std::vector<Run> runs;
            for (Lane& l : call.lanes) {
                const int n_lane = l.f_end - l.f_begin;
                for (int i = 0; i < n_lane;) {
                    if (!l.h_flags[i]) { ++i; continue; }
                    int e = i;
                    while (e < n_lane && l.h_flags[e]) ++e;
                    runs.push_back(Run{&l, l.f_begin + i, l.f_begin + e});
                    i = e;
                }
            }
            for (const Run& r : runs) {
                if ((rc = call.use(*r.l))) return rc;
                const int hc2 = host_chunk_frames(rows, cols, r.e - r.f);
                const size_t bytes2 = 2 * carve_bytes(fpix * hc2, sizeof(float)) + (guided ? carve_bytes(fpix * hc2, sizeof(int32_t)) : 0) +
                                      carve_bytes((size_t)hc2 * DCMT_STATS_STRIDE, sizeof(int32_t)) + carve_bytes((size_t)hc2, sizeof(int32_t)) +
                                      completion_ws_bytes(rows, cols, hc2, bilateral, lf, false, lf);
                for (int f = r.f; f < r.e; f += hc2)
                    if ((rc = do_chunk(*r.l, f, std::min(hc2, r.e - f), cg, lf, hc2, bytes2))) return rc;
                any = true;
            }
            if (any && (rc = call.finish())) return rc;
            if (level == DCMT_PATH_GENERIC || !any) break;
        }
    }
    return DCMT_OK;
}

// ---- KITTI uint16 input (main.cpp:75-82: imread(IMREAD_ANYDEPTH) + convertTo(CV_32F, 1/256) + img_completion) ----
int validate_completion_u16(const uint16_t* sparse, float* dense, int rows, int cols, size_t in_pitch_bytes,
                            size_t in_frame_stride_bytes, size_t out_pitch_bytes, size_t out_frame_stride_bytes, int n_frames,
                            int blur_type, int flags, Geometry* gi, Geometry* go) {
    if (!sparse || !dense) return fail(DCMT_E_BADARG, "null image pointer");
    if (blur_type < DCMT_BLUR_NONE || blur_type > DCMT_BLUR_BILATERAL) return fail(DCMT_E_BADARG, "blur_type %d", blur_type);
    if (flags < DCMT_PATH_AUTO || flags > DCMT_PATH_RANK) return fail(DCMT_E_BADARG, "flags %d", flags);
    int rc = check_geometry(rows, cols, in_pitch_bytes, in_frame_stride_bytes, n_frames, gi, sizeof(uint16_t));
    if (rc) return rc;
    if ((rc = check_geometry(rows, cols, out_pitch_bytes, out_frame_stride_bytes, n_frames, go, sizeof(float)))) return rc;
    if (n_frames && overlaps(sparse, gi->span_bytes, dense, go->span_bytes)) return fail(DCMT_E_BADARG, "input and output overlap");
    return DCMT_OK;
}

int run_completion_u16(const uint16_t* sparse, float* dense, int rows, int cols, size_t in_pitch_bytes,
                       size_t in_frame_stride_bytes, size_t out_pitch_bytes, size_t out_frame_stride_bytes, int n_frames,
                       int blur_type, int flags, int32_t* stats, cudaStream_t st) {
    Geometry gi, go;
    int rc = validate_completion_u16(sparse, dense, rows, cols, in_pitch_bytes, in_frame_stride_bytes, out_pitch_bytes,
                                     out_frame_stride_bytes, n_frames, blur_type, flags, &gi, &go);
    if (rc) return rc;
    if (n_frames == 0) return DCMT_OK;
    if ((rc = check_device())) return rc;
    API_CUDA(dcmt::generic_configure(), "kernel attribute setup");
    API_CUDA(dcmt::q8_configure(), "kernel attribute setup");
    // uint16 input needs no validation: AUTO and FUSED are the same thing here
    CompletionCall cc{nullptr, 0, false, rows, cols, blur_type, flags == DCMT_PATH_GENERIC ? DCMT_PATH_GENERIC : DCMT_PATH_FUSED};
    const bool fused = fused_applies(cc);
    Arena* ar = nullptr;
    if ((rc = arena_acquire(st, completion_ws_bytes(rows, cols, n_frames, blur_type == DCMT_BLUR_BILATERAL, fused, true), &ar))) return rc;
    return enqueue_completion(cc, nullptr, nullptr, dense, go.pitch, go.fstride, n_frames, stats, nullptr, nullptr, nullptr, ar, st,
                              nullptr, U16Input{sparse, gi.pitch, gi.fstride});
}

int run_completion_u16_host(const uint16_t* sparse, float* dense, int rows, int cols, size_t in_pitch_bytes,
                            size_t in_frame_stride_bytes, size_t out_pitch_bytes, size_t out_frame_stride_bytes, int n_frames,
                            int blur_type, int flags, int32_t* stats, const int* devices = nullptr, int n_devices = 0, bool multi = false,
                            bool copy_only = false) {
    Geometry gi, go;
    int rc = validate_completion_u16(sparse, dense, rows, cols, in_pitch_bytes, in_frame_stride_bytes, out_pitch_bytes,
                                     out_frame_stride_bytes, n_frames, blur_type, flags, &gi, &go);
    if (rc) return rc;
    if (n_frames == 0) return DCMT_OK;
    HostCall call;
    if ((rc = call.open(devices, n_devices, multi))) return rc;
    call.split(n_frames);
    const size_t fpix = (size_t)rows * cols;
    const size_t in_pitch = ((size_t)cols + 7) / 8 * 8;  // device rows 16-byte aligned: vector loads in k_q8_front
    int longest = 0;
    for (Lane& l : call.lanes) longest = std::max(longest, l.f_end - l.f_begin);
    const int hc = host_chunk_frames(rows, cols, longest);
    CompletionCall cc{nullptr, 0, false, rows, cols, blur_type, flags == DCMT_PATH_GENERIC ? DCMT_PATH_GENERIC : DCMT_PATH_FUSED};
    const bool fused = fused_applies(cc);
    const size_t bytes = carve_bytes((size_t)rows * in_pitch * hc, sizeof(uint16_t)) + carve_bytes(fpix * hc, sizeof(float)) +
                         carve_bytes((size_t)hc * DCMT_STATS_STRIDE, sizeof(int32_t)) +
                         completion_ws_bytes(rows, cols, hc, blur_type == DCMT_BLUR_BILATERAL, fused, true);
    for (Lane& l : call.lanes) {
        if (l.f_end == l.f_begin) continue;
        if ((rc = call.use(l))) return rc;
        API_CUDA(dcmt::generic_configure(), "kernel attribute setup");
        API_CUDA(dcmt::q8_configure(), "kernel attribute setup");
    }
    for (bool more = true; more;) {
        more = false;
        for (Lane& l : call.lanes) {
            if (l.next >= l.f_end) continue;
            more = true;
            if ((rc = call.use(l))) return rc;
            const int f0 = l.next, nf = std::min(hc, l.f_end - f0);
            l.next += nf;
            cudaStream_t st = l.hs->s[l.slot];
            l.slot = (l.slot + 1) % kHostStreams;
            Arena* ar = nullptr;
            if ((rc = arena_acquire(st, bytes, &ar))) return rc;
            uint16_t* d_in = carve<uint16_t>(ar, (size_t)rows * in_pitch * hc);
            float* d_out = carve<float>(ar, fpix * hc);
            int32_t* d_stats = carve<int32_t>(ar, (size_t)hc * DCMT_STATS_STRIDE);
            if ((rc = arena_ok(ar))) return rc;
            if ((rc = copy_frames_h2d(d_in, in_pitch * sizeof(uint16_t), sparse + (size_t)f0 * gi.fstride, gi.pitch * sizeof(uint16_t),
                                      gi.fstride * sizeof(uint16_t), (size_t)cols * sizeof(uint16_t), rows, nf, st)))
                return rc;
            if (copy_only) {
                API_CUDA(cudaMemsetAsync(d_out, 0, fpix * nf * sizeof(float), st), "memset");
            } else if ((rc = enqueue_completion(cc, nullptr, nullptr, d_out, cols, fpix, nf, stats ? d_stats : nullptr, nullptr, nullptr,
                                                nullptr, ar, st, nullptr, U16Input{d_in, in_pitch, (size_t)rows * in_pitch}))) {
                return rc;
            }
            if ((rc = copy_frames_d2h(dense + (size_t)f0 * go.fstride, go.pitch * sizeof(float), go.fstride * sizeof(float), d_out,
                                      (size_t)cols * sizeof(float), rows, nf, st)))
                return rc;
            if (stats && !copy_only)
                API_CUDA(cudaMemcpyAsync(stats + (size_t)f0 * DCMT_STATS_STRIDE, d_stats, (size_t)nf * DCMT_STATS_STRIDE * sizeof(int32_t),
                                         cudaMemcpyDeviceToHost, st),
                         "device to host copy");
        }
    }
    return call.finish();
}

}  // namespace

extern "C" {

static int check_planes(int rows, int cols, int n_frames);

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
    return completion_ws_bytes(rows, cols, n_frames, true, true, true, true);  // upper bound over the paths a call may take
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
    return run_completion(sparse, nullptr, 0, false, dense, rows, cols, pitch_bytes, frame_stride_bytes, n_frames, blur_type,
                          flags, stats, nullptr, nullptr, static_cast<cudaStream_t>(cuda_stream));
}

int dcmt_img_completion_f32_host(const float* sparse, float* dense, int rows, int cols, size_t pitch_bytes,
                                 size_t frame_stride_bytes, int n_frames, int blur_type, int flags, int32_t* stats) {
    return run_completion_host(sparse, nullptr, 0, false, dense, rows, cols, pitch_bytes, frame_stride_bytes, n_frames,
                               blur_type, flags, stats);
}

int dcmt_img_completion_u16(const uint16_t* sparse_u16, float* dense, int rows, int cols, size_t in_pitch_bytes,
                            size_t in_frame_stride_bytes, size_t out_pitch_bytes, size_t out_frame_stride_bytes, int n_frames,
                            int blur_type, int flags, int32_t* stats, void* cuda_stream) {
    return run_completion_u16(sparse_u16, dense, rows, cols, in_pitch_bytes, in_frame_stride_bytes, out_pitch_bytes,
                              out_frame_stride_bytes, n_frames, blur_type, flags, stats, static_cast<cudaStream_t>(cuda_stream));
}

int dcmt_img_completion_u16_host(const uint16_t* sparse_u16, float* dense, int rows, int cols, size_t in_pitch_bytes,
                                 size_t in_frame_stride_bytes, size_t out_pitch_bytes, size_t out_frame_stride_bytes,
                                 int n_frames, int blur_type, int flags, int32_t* stats) {
    return run_completion_u16_host(sparse_u16, dense, rows, cols, in_pitch_bytes, in_frame_stride_bytes, out_pitch_bytes,
                                   out_frame_stride_bytes, n_frames, blur_type, flags, stats);
}

int dcmt_img_completion_f32_host_multi(const float* sparse, float* dense, int rows, int cols, size_t pitch_bytes,
                                       size_t frame_stride_bytes, int n_frames, int blur_type, int flags, int32_t* stats,
                                       const int* devices, int n_devices) {
    return run_completion_host(sparse, nullptr, 0, false, dense, rows, cols, pitch_bytes, frame_stride_bytes, n_frames,
                               blur_type, flags, stats, devices, n_devices, true);
}

int dcmt_img_completion_u16_host_multi(const uint16_t* sparse_u16, float* dense, int rows, int cols, size_t in_pitch_bytes,
                                       size_t in_frame_stride_bytes, size_t out_pitch_bytes, size_t out_frame_stride_bytes,
                                       int n_frames, int blur_type, int flags, int32_t* stats, const int* devices, int n_devices) {
    return run_completion_u16_host(sparse_u16, dense, rows, cols, in_pitch_bytes, in_frame_stride_bytes, out_pitch_bytes,
                                   out_frame_stride_bytes, n_frames, blur_type, flags, stats, devices, n_devices, true);
}

int dcmt_interpolate_with_superpixels_f32_host_multi(const float* sparse, const int32_t* labels, int n_clusters, float* dense, int rows,
                                                     int cols, size_t pitch_bytes, size_t frame_stride_bytes, int n_frames,
                                                     int use_superpixel, int flags, int32_t* stats, const int* devices, int n_devices) {
    return run_completion_host(sparse, labels, n_clusters, use_superpixel != 0, dense, rows, cols, pitch_bytes, frame_stride_bytes,
                               n_frames, DCMT_BLUR_GAUSSIAN, flags, stats, devices, n_devices, true);
}

int dcmt_debug_host_copy_f32(const float* in, float* out, int rows, int cols, int n_frames, const int* devices, int n_devices) {
    return run_completion_host(in, nullptr, 0, false, out, rows, cols, 0, 0, n_frames, DCMT_BLUR_NONE, DCMT_PATH_AUTO, nullptr, devices,
                               n_devices, devices != nullptr || n_devices != 0, true);
}

int dcmt_debug_host_copy_u16(const uint16_t* in, float* out, int rows, int cols, int n_frames, const int* devices, int n_devices) {
    return run_completion_u16_host(in, out, rows, cols, 0, 0, 0, 0, n_frames, DCMT_BLUR_NONE, DCMT_PATH_AUTO, nullptr, devices, n_devices,
                                   devices != nullptr || n_devices != 0, true);
}

int dcmt_interpolate_with_superpixels_ex_f32(const float* sparse, const int32_t* labels, int n_clusters, float* dense, int rows,
                                             int cols, size_t pitch_bytes, size_t frame_stride_bytes, int n_frames, int use_superpixel,
                                             int flags, int32_t* stats, void* cuda_stream) {
    // blur is unconditionally Gaussian in the reference (img_completion_lc.cpp:183-192)
    return run_completion(sparse, labels, n_clusters, use_superpixel != 0, dense, rows, cols, pitch_bytes, frame_stride_bytes,
                          n_frames, DCMT_BLUR_GAUSSIAN, flags, stats, nullptr, nullptr, static_cast<cudaStream_t>(cuda_stream));
}

int dcmt_interpolate_with_superpixels_ex_f32_host(const float* sparse, const int32_t* labels, int n_clusters, float* dense, int rows,
                                                  int cols, size_t pitch_bytes, size_t frame_stride_bytes, int n_frames,
                                                  int use_superpixel, int flags, int32_t* stats) {
    return run_completion_host(sparse, labels, n_clusters, use_superpixel != 0, dense, rows, cols, pitch_bytes, frame_stride_bytes,
                               n_frames, DCMT_BLUR_GAUSSIAN, flags, stats);
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
    int rc = run_completion(sparse, nullptr, 0, false, dense, rows, cols, 0, 0, 1, blur_type, DCMT_PATH_GENERIC, nullptr,
                            stages, &mask, static_cast<cudaStream_t>(cuda_stream));
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
    Arena* ar = nullptr;
    const size_t fpix = (size_t)rows * cols;
    const size_t mid_pitch = ((size_t)cols + 7) / 8 * 8;
    const size_t bytes = 2 * carve_bytes(fpix * n_frames, 4) + carve_bytes(n_frames, sizeof(dcmt::FrameCounters)) +
                         carve_bytes((size_t)rows * mid_pitch * n_frames, 2) + 2 * carve_bytes(mid_pitch * n_frames, 4);
    if ((rc = arena_acquire(st, bytes, &ar))) return rc;
    dcmt::Q8Plan p{};
    p.rows = rows;
    p.cols = cols;
    dcmt::q8_choose_tile(rows, cols, &p.th, &p.tw);
    p.mid_pitch = (int)mid_pitch;
    p.max_frames = n_frames;
    p.w1 = carve<float>(ar, fpix * n_frames);
    p.w2 = carve<float>(ar, fpix * n_frames);
    p.ctr = carve<dcmt::FrameCounters>(ar, n_frames);
    p.mid = carve<uint16_t>(ar, (size_t)rows * mid_pitch * n_frames);
    p.col_first = carve<uint32_t>(ar, mid_pitch * n_frames);
    p.col_last = carve<uint32_t>(ar, mid_pitch * n_frames);
    if ((rc = arena_ok(ar))) return rc;
    p.prof_front = front_stamps;
    p.prof_tail = tail_stamps;
    if (tiles_per_frame) *tiles_per_frame = ((cols + p.tw - 1) / p.tw) * ((rows + p.th - 1) / p.th);
    API_CUDA(dcmt::q8_run_front(p, sparse, nullptr, cols, fpix, n_frames, 1, st), "fused front launch");
    API_CUDA(dcmt::q8_run_tail(p, dense, cols, fpix, n_frames, DCMT_BLUR_GAUSSIAN, st), "fused tail launch");
    return DCMT_OK;
}

int dcmt_slic_center_count(int rows, int cols, int step) {
    if (rows < 1 || cols < 1 || step < 1) return 0;
    return dcmt::slic_center_count(rows, cols, step);
}

// Slic::generate_superpixels on the Lab image `img`, or, with from_bgr, on the cvtColor(COLOR_BGR2Lab) of the BGR image
// `img`: the Lab frames then live in the SLIC workspace of (device, stream) and never leave the device
static int slic_device(const uint8_t* img, bool from_bgr, int rows, int cols, int n_frames, int step, int nc, int iterations,
                       int32_t* labels, double* centers, void* cuda_stream) {
    if (!img || !labels) return fail(DCMT_E_BADARG, "null pointer");
    int rc = check_planes(rows, cols, n_frames);
    if (rc) return rc;
    if (nc == 0 || iterations < 0) return fail(DCMT_E_BADARG, "nc %d, iterations %d", nc, iterations);
    if (step < 4) return fail(DCMT_E_UNSUPPORTED, "step %d: find_local_minimum (slic.cpp:72-99) reads outside the image below 4", step);
    if (rows >= 1 << 24 || cols >= 1 << 24) return fail(DCMT_E_UNSUPPORTED, "SLIC frames are limited to 2^24 rows / columns");
    if ((size_t)rows * (size_t)cols > (size_t)1 << 30) return fail(DCMT_E_UNSUPPORTED, "frame larger than 2^30 pixels");
    if (n_frames > 65535) return fail(DCMT_E_UNSUPPORTED, "at most 65535 frames per call");
    if (n_frames == 0) return DCMT_OK;
    if ((rc = check_device())) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    const int k = dcmt::slic_center_count(rows, cols, step);
    dcmt::SlicWork w{};
    const size_t nbins = dcmt::slic_bins(rows, cols, step, &w.bins_x, &w.bins_y);
    const size_t kk = (k > 0 ? (size_t)k : 1) * n_frames, nb = nbins * n_frames;
    Arena* ar = nullptr;
    if ((rc = arena_acquire(st, 2 * carve_bytes(kk * 5, sizeof(double)) + carve_bytes(kk * 6, sizeof(unsigned long long)) +
                                    carve_bytes(nb + n_frames, sizeof(int)) + carve_bytes(nb, sizeof(int)) + carve_bytes(kk, sizeof(int)) +
                                    (from_bgr ? carve_bytes((size_t)rows * cols * 3 * n_frames, 1) : 0),
                            &ar)))
        return rc;
    w.centers = carve<double>(ar, kk * 5);
    w.sums = carve<unsigned long long>(ar, kk * 6);
    w.bin_count = carve<int>(ar, nb + n_frames);
    w.bin_fill = carve<int>(ar, nb);
    w.bin_items = carve<int>(ar, kk);
    w.sorted = carve<double>(ar, kk * 5);
    uint8_t* lab = from_bgr ? carve<uint8_t>(ar, (size_t)rows * cols * 3 * n_frames) : nullptr;
    if ((rc = arena_ok(ar))) return rc;
    if (from_bgr) {
        const size_t pitch = (size_t)cols * 3;
        API_CUDA(dcmt::color_bgr2lab(img, pitch, pitch * rows, lab, pitch, pitch * rows, rows, cols, n_frames, st), "BGR2Lab launch");
    }
    API_CUDA(dcmt::slic_run(from_bgr ? lab : img, rows, cols, n_frames, step, nc, iterations, labels, k, w, st), "SLIC launch");
    if (centers && k > 0)
        API_CUDA(cudaMemcpyAsync(centers, w.centers, (size_t)k * n_frames * 5 * sizeof(double), cudaMemcpyDeviceToDevice, st), "centre copy");
    return DCMT_OK;
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
    if (!img || !labels) return fail(DCMT_E_BADARG, "null pointer");
    int rc = check_planes(rows, cols, n_frames);
    if (rc) return rc;
    if (n_frames == 0) return DCMT_OK;
    HostCall call;
    if ((rc = call.open(nullptr, 0, false))) return rc;
    // staging buffers come from the arena of an internal stream (no cudaMalloc per call), copies are asynchronous on it
    cudaStream_t st = call.lanes[0].hs->s[0];
    const size_t n = (size_t)rows * cols * n_frames;
    const size_t k = (size_t)(step >= 1 ? dcmt::slic_center_count(rows, cols, step) : 0) * n_frames;
    Arena* stage = nullptr;
    {
        // a second arena key on the same device: the SLIC work arena is keyed by `st`, the staging one by the next stream
        cudaStream_t st2 = call.lanes[0].hs->s[1];
        if ((rc = arena_acquire(st2, carve_bytes(n * 3, 1) + carve_bytes(n, 4) + carve_bytes((k > 0 ? k : 1) * 5, sizeof(double)), &stage))) return rc;
    }
    uint8_t* d_img = carve<uint8_t>(stage, n * 3);
    int32_t* d_labels = carve<int32_t>(stage, n);
    double* d_centers = carve<double>(stage, (k > 0 ? k : 1) * 5);
    if ((rc = arena_ok(stage))) return rc;
    call.use(call.lanes[0]);
    API_CUDA(cudaMemcpyAsync(d_img, img, n * 3, cudaMemcpyHostToDevice, st), "host to device copy");
    if ((rc = slic_device(d_img, from_bgr, rows, cols, n_frames, step, nc, iterations, d_labels, centers ? d_centers : nullptr, st))) return rc;
    API_CUDA(cudaMemcpyAsync(labels, d_labels, n * 4, cudaMemcpyDeviceToHost, st), "device to host copy");
    if (centers && k > 0) API_CUDA(cudaMemcpyAsync(centers, d_centers, k * 5 * sizeof(double), cudaMemcpyDeviceToHost, st), "device to host copy");
    return call.finish();
}

int dcmt_slic_u8c3_host(const uint8_t* lab, int rows, int cols, int n_frames, int step, int nc, int iterations, int32_t* labels,
                        double* centers) {
    return slic_host(lab, false, rows, cols, n_frames, step, nc, iterations, labels, centers);
}

int dcmt_slic_bgr_u8c3_host(const uint8_t* bgr, int rows, int cols, int n_frames, int step, int nc, int iterations, int32_t* labels,
                            double* centers) {
    return slic_host(bgr, true, rows, cols, n_frames, step, nc, iterations, labels, centers);
}

int dcmt_lidar_project_f32(const float* points, int n_points, const float* T_host, const float* P_host, int rows, int cols,
                           float* projected, float* normalized, float norm_a, float norm_b, int32_t* n_projected, void* cuda_stream) {
    if ((!points && n_points > 0) || !T_host || !P_host) return fail(DCMT_E_BADARG, "null pointer");
    if (n_points < 0) return fail(DCMT_E_BADARG, "n_points must be >= 0 (got %d)", n_points);
    int rc = check_planes(rows, cols, 1);
    if (rc) return rc;
    if ((size_t)rows * (size_t)cols > (size_t)1 << 30) return fail(DCMT_E_UNSUPPORTED, "frame larger than 2^30 pixels");
    if (points && (reinterpret_cast<uintptr_t>(points) & 15)) return fail(DCMT_E_BADARG, "points must be 16-byte aligned");
    if ((rc = check_device())) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    Arena* ar = nullptr;
    const size_t nk = dcmt::project_key_count(rows, cols);
    if ((rc = arena_acquire(st, carve_bytes(nk, sizeof(unsigned long long)) + carve_bytes(8, sizeof(unsigned)), &ar))) return rc;
    dcmt::ProjectWork w{carve<unsigned long long>(ar, nk), carve<unsigned>(ar, 8)};
    if ((rc = arena_ok(ar))) return rc;
    API_CUDA(dcmt::project_run(points, n_points, T_host, P_host, rows, cols, projected, normalized, norm_a, norm_b, n_projected, w, st),
             "projection launch");
    return DCMT_OK;
}

int dcmt_lidar_project_batch_f32(const float* points, const int32_t* n_points_dev_or_null, int max_points, size_t cloud_stride_points,
                                 int n_clouds, const float* T_host, const float* P_host, int rows, int cols, float* projected,
                                 float* normalized, float norm_a, float norm_b, int32_t* n_projected, void* cuda_stream) {
    if ((!points && max_points > 0) || !T_host || !P_host) return fail(DCMT_E_BADARG, "null pointer");
    if (max_points < 0 || n_clouds < 0) return fail(DCMT_E_BADARG, "max_points %d, n_clouds %d", max_points, n_clouds);
    if (n_clouds > 65535) return fail(DCMT_E_UNSUPPORTED, "at most 65535 clouds per call");
    if (n_clouds > 1 && cloud_stride_points < (size_t)max_points) return fail(DCMT_E_BADARG, "cloud_stride_points %zu < max_points %d", cloud_stride_points, max_points);
    int rc = check_planes(rows, cols, 1);
    if (rc) return rc;
    if ((size_t)rows * (size_t)cols > (size_t)1 << 30) return fail(DCMT_E_UNSUPPORTED, "frame larger than 2^30 pixels");
    if (points && (reinterpret_cast<uintptr_t>(points) & 15)) return fail(DCMT_E_BADARG, "points must be 16-byte aligned");
    if (n_clouds == 0) return DCMT_OK;
    if ((rc = check_device())) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    Arena* ar = nullptr;
    const size_t nk = dcmt::project_key_count(rows, cols) * n_clouds;
    if ((rc = arena_acquire(st, carve_bytes(nk, sizeof(unsigned long long)) + carve_bytes(8 * (size_t)n_clouds, sizeof(unsigned)), &ar))) return rc;
    dcmt::ProjectWork w{carve<unsigned long long>(ar, nk), carve<unsigned>(ar, 8 * (size_t)n_clouds)};
    if ((rc = arena_ok(ar))) return rc;
    API_CUDA(dcmt::project_run_batch(points, max_points, n_points_dev_or_null, cloud_stride_points, n_clouds, T_host, P_host, rows, cols,
                                     projected, normalized, norm_a, norm_b, n_projected, w, st),
             "projection launch");
    return DCMT_OK;
}

int dcmt_lidar_project_f32_host(const float* points, int n_points, const float* T_host, const float* P_host, int rows, int cols,
                                float* projected, float* normalized, float norm_a, float norm_b, int32_t* n_projected) {
    if ((!points && n_points > 0) || !T_host || !P_host) return fail(DCMT_E_BADARG, "null pointer");
    if (n_points < 0) return fail(DCMT_E_BADARG, "n_points must be >= 0 (got %d)", n_points);
    int rc = check_planes(rows, cols, 1);
    if (rc) return rc;
    HostCall call;
    if ((rc = call.open(nullptr, 0, false))) return rc;
    cudaStream_t st = call.lanes[0].hs->s[0], st2 = call.lanes[0].hs->s[1];
    const size_t n = (size_t)rows * cols;
    Arena* stage = nullptr;
    if ((rc = arena_acquire(st2, carve_bytes((size_t)(n_points > 0 ? n_points : 1) * 4, 4) + 2 * carve_bytes(n, 4) + carve_bytes(1, 4), &stage)))
        return rc;
    float* d_pts = carve<float>(stage, (size_t)(n_points > 0 ? n_points : 1) * 4);
    float* d_proj = carve<float>(stage, n);
    float* d_norm = carve<float>(stage, n);
    int32_t* d_cnt = carve<int32_t>(stage, 1);
    if ((rc = arena_ok(stage))) return rc;
    call.use(call.lanes[0]);
    if (n_points > 0) API_CUDA(cudaMemcpyAsync(d_pts, points, (size_t)n_points * 16, cudaMemcpyHostToDevice, st), "host to device copy");
    if ((rc = dcmt_lidar_project_f32(d_pts, n_points, T_host, P_host, rows, cols, d_proj, d_norm, norm_a, norm_b, d_cnt, st))) return rc;
    if (projected) API_CUDA(cudaMemcpyAsync(projected, d_proj, n * 4, cudaMemcpyDeviceToHost, st), "device to host copy");
    if (normalized) API_CUDA(cudaMemcpyAsync(normalized, d_norm, n * 4, cudaMemcpyDeviceToHost, st), "device to host copy");
    if (n_projected) API_CUDA(cudaMemcpyAsync(n_projected, d_cnt, 4, cudaMemcpyDeviceToHost, st), "device to host copy");
    return call.finish();
}

static_assert(sizeof(dcmt_eval_result) == sizeof(dcmt::EvalResult), "dcmt_eval_result and dcmt::EvalResult must match");

int dcmt_evaluate_f32(const float* gt, const float* dense, int rows, int cols, size_t pitch_bytes, size_t frame_stride_bytes,
                      int n_frames, float tolerance, int mode, dcmt_eval_result* results, void* cuda_stream) {
    if (!gt || !dense || !results) return fail(DCMT_E_BADARG, "null pointer");
    if (mode != DCMT_EVAL_GT_VALID && mode != DCMT_EVAL_BOTH_VALID) return fail(DCMT_E_BADARG, "mode %d", mode);
    Geometry g;
    int rc = check_geometry(rows, cols, pitch_bytes, frame_stride_bytes, n_frames, &g);
    if (rc) return rc;
    if (n_frames == 0) return DCMT_OK;
    if ((rc = check_device())) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    Arena* ar = nullptr;
    if ((rc = arena_acquire(st, carve_bytes(dcmt::eval_partial_doubles(n_frames), sizeof(double)), &ar))) return rc;
    double* partials = carve<double>(ar, dcmt::eval_partial_doubles(n_frames));
    if ((rc = arena_ok(ar))) return rc;
    API_CUDA(dcmt::eval_run(gt, dense, rows, cols, g.pitch, g.fstride, n_frames, tolerance, mode, partials,
                            reinterpret_cast<dcmt::EvalResult*>(results), st),
             "evaluation launch");
    return DCMT_OK;
}

int dcmt_evaluate_f32_host(const float* gt, const float* dense, int rows, int cols, size_t pitch_bytes, size_t frame_stride_bytes,
                           int n_frames, float tolerance, int mode, dcmt_eval_result* results) {
    if (!gt || !dense || !results) return fail(DCMT_E_BADARG, "null pointer");
    if (mode != DCMT_EVAL_GT_VALID && mode != DCMT_EVAL_BOTH_VALID) return fail(DCMT_E_BADARG, "mode %d", mode);
    Geometry g;
    int rc = check_geometry(rows, cols, pitch_bytes, frame_stride_bytes, n_frames, &g);
    if (rc) return rc;
    if (n_frames == 0) return DCMT_OK;
    HostCall call;
    if ((rc = call.open(nullptr, 0, false))) return rc;
    cudaStream_t st = call.lanes[0].hs->s[0], st2 = call.lanes[0].hs->s[1];
    Arena* stage = nullptr;
    if ((rc = arena_acquire(st2, 2 * carve_bytes(g.span_bytes, 1) + carve_bytes((size_t)n_frames, sizeof(dcmt_eval_result)), &stage))) return rc;
    float* d_gt = reinterpret_cast<float*>(carve<char>(stage, g.span_bytes));
    float* d_r = reinterpret_cast<float*>(carve<char>(stage, g.span_bytes));
    dcmt_eval_result* d_res = carve<dcmt_eval_result>(stage, (size_t)n_frames);
    if ((rc = arena_ok(stage))) return rc;
    call.use(call.lanes[0]);
    API_CUDA(cudaMemcpyAsync(d_gt, gt, g.span_bytes, cudaMemcpyHostToDevice, st), "host to device copy");
    API_CUDA(cudaMemcpyAsync(d_r, dense, g.span_bytes, cudaMemcpyHostToDevice, st), "host to device copy");
    if ((rc = dcmt_evaluate_f32(d_gt, d_r, rows, cols, pitch_bytes, frame_stride_bytes, n_frames, tolerance, mode, d_res, st))) return rc;
    API_CUDA(cudaMemcpyAsync(results, d_res, (size_t)n_frames * sizeof(dcmt_eval_result), cudaMemcpyDeviceToHost, st), "device to host copy");
    return call.finish();
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

static int check_planes(int rows, int cols, int n_frames) {
    if (rows < 1 || cols < 1) return fail(DCMT_E_BADARG, "rows and cols must be >= 1 (got %d x %d)", rows, cols);
    if (n_frames < 0) return fail(DCMT_E_BADARG, "n_frames must be >= 0 (got %d)", n_frames);
    return DCMT_OK;
}

int dcmt_stereo_refine_f32(const float* depth_ig, const uint8_t* left_gray, const uint8_t* right_gray, float* depth_out,
                           float* disp_out, int rows, int cols, int n_frames, const dcmt_stereo_params* prm,
                           void* cuda_stream) {
    if (!depth_ig || !left_gray || !right_gray || !depth_out || !prm) return fail(DCMT_E_BADARG, "null pointer");
    int rc = check_planes(rows, cols, n_frames);
    if (rc) return rc;
    if (prm->num_iterations < 0) return fail(DCMT_E_BADARG, "num_iterations %d", prm->num_iterations);
    if ((size_t)rows * (size_t)cols > (size_t)1 << 30) return fail(DCMT_E_UNSUPPORTED, "frame larger than 2^30 pixels");
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
    if (!depth_ig || !left_gray || !right_gray || !depth_out || !prm) return fail(DCMT_E_BADARG, "null pointer");
    int rc = check_planes(rows, cols, n_frames);
    if (rc) return rc;
    if (prm->num_iterations < 0) return fail(DCMT_E_BADARG, "num_iterations %d", prm->num_iterations);
    if ((size_t)rows * (size_t)cols > (size_t)1 << 30) return fail(DCMT_E_UNSUPPORTED, "frame larger than 2^30 pixels");
    if (n_frames == 0) return DCMT_OK;
    // chunks of frames flow H2D -> kernel -> D2H round-robin over the three host streams (asynchronous for page-locked buffers)
    HostCall call;
    if ((rc = call.open(nullptr, 0, false))) return rc;
    HostStreams* hs = call.lanes[0].hs;
    call.use(call.lanes[0]);
    const size_t fpix = (size_t)rows * cols;
    const int hc = host_chunk_frames(rows, cols, n_frames);
    const size_t bytes = 2 * carve_bytes(fpix * hc, sizeof(float)) + (disp_out ? carve_bytes(fpix * hc, sizeof(float)) : 0) +
                         2 * carve_bytes(fpix * hc, sizeof(uint8_t));
    int slot = 0;
    for (int f0 = 0; f0 < n_frames; f0 += hc, slot = (slot + 1) % kHostStreams) {
        const int nf = n_frames - f0 < hc ? n_frames - f0 : hc;
        cudaStream_t st = hs->s[slot];
        Arena* ar = nullptr;
        if ((rc = arena_acquire(st, bytes, &ar))) return rc;
        float* d_ig = carve<float>(ar, fpix * hc);
        float* d_out = carve<float>(ar, fpix * hc);
        float* d_disp = disp_out ? carve<float>(ar, fpix * hc) : nullptr;
        uint8_t* d_l = carve<uint8_t>(ar, fpix * hc);
        uint8_t* d_r = carve<uint8_t>(ar, fpix * hc);
        if ((rc = arena_ok(ar))) return rc;
        const size_t off = (size_t)f0 * fpix, n = fpix * nf;
        API_CUDA(cudaMemcpyAsync(d_ig, depth_ig + off, n * 4, cudaMemcpyHostToDevice, st), "host to device copy");
        API_CUDA(cudaMemcpyAsync(d_l, left_gray + off, n, cudaMemcpyHostToDevice, st), "host to device copy");
        API_CUDA(cudaMemcpyAsync(d_r, right_gray + off, n, cudaMemcpyHostToDevice, st), "host to device copy");
        if ((rc = dcmt_stereo_refine_f32(d_ig, d_l, d_r, d_out, d_disp, rows, cols, nf, prm, st))) return rc;
        API_CUDA(cudaMemcpyAsync(depth_out + off, d_out, n * 4, cudaMemcpyDeviceToHost, st), "device to host copy");
        if (disp_out) API_CUDA(cudaMemcpyAsync(disp_out + off, d_disp, n * 4, cudaMemcpyDeviceToHost, st), "device to host copy");
    }
    return call.finish();
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
    HostCall call;
    if ((rc = call.open(nullptr, 0, false))) return rc;
    cudaStream_t st = call.lanes[0].hs->s[0];
    const size_t in_row = (size_t)cols * 3, frames_rows = (size_t)rows * n_frames;
    Arena* ar = nullptr;
    if ((rc = arena_acquire(st, carve_bytes(in_row * frames_rows, 1) + carve_bytes((size_t)cols * frames_rows, 1), &ar))) return rc;
    uint8_t* d_in = carve<uint8_t>(ar, in_row * frames_rows);
    uint8_t* d_out = carve<uint8_t>(ar, (size_t)cols * frames_rows);
    if ((rc = arena_ok(ar))) return rc;
    call.use(call.lanes[0]);
    API_CUDA(cudaMemcpy2DAsync(d_in, in_row, bgr, bgr_pitch_bytes, in_row, frames_rows, cudaMemcpyHostToDevice, st), "host to device copy");
    if ((rc = dcmt_bgr2gray_u8(d_in, d_out, rows, cols, 0, 0, n_frames, st))) return rc;
    API_CUDA(cudaMemcpy2DAsync(gray, gray_pitch_bytes, d_out, cols, cols, frames_rows, cudaMemcpyDeviceToHost, st), "device to host copy");
    return call.finish();
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
    HostCall call;
    if ((rc = call.open(nullptr, 0, false))) return rc;
    cudaStream_t st = call.lanes[0].hs->s[0];
    const size_t row = (size_t)cols * 3, frames_rows = (size_t)rows * n_frames;
    Arena* ar = nullptr;
    if ((rc = arena_acquire(st, 2 * carve_bytes(row * frames_rows, 1), &ar))) return rc;
    uint8_t* d_in = carve<uint8_t>(ar, row * frames_rows);
    uint8_t* d_out = carve<uint8_t>(ar, row * frames_rows);
    if ((rc = arena_ok(ar))) return rc;
    call.use(call.lanes[0]);
    API_CUDA(cudaMemcpy2DAsync(d_in, row, bgr, bgr_pitch_bytes, row, frames_rows, cudaMemcpyHostToDevice, st), "host to device copy");
    if ((rc = dcmt_bgr2lab_u8(d_in, d_out, rows, cols, 0, 0, n_frames, st))) return rc;
    API_CUDA(cudaMemcpy2DAsync(lab, lab_pitch_bytes, d_out, row, row, frames_rows, cudaMemcpyDeviceToHost, st), "device to host copy");
    return call.finish();
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

int dcmt_entries_optimize_ig(const void* entries_left, size_t left_row_step_bytes, const void* entries_right, size_t right_row_step_bytes,
                             size_t elem_stride_bytes, float* disp, size_t disp_pitch_bytes, int rows, int cols, int num_iterations,
                             float damp_factor, float err_clip, void* cuda_stream) {
    int rc = check_entries(entries_left, rows, cols, left_row_step_bytes, elem_stride_bytes);
    if (rc) return rc;
    if ((rc = check_entries(entries_right, rows, cols, right_row_step_bytes, elem_stride_bytes))) return rc;
    if ((rc = check_mat_f32(disp, rows, cols, &disp_pitch_bytes))) return rc;
    if (num_iterations < 0) return fail(DCMT_E_BADARG, "num_iterations %d", num_iterations);
    if ((rc = check_device())) return rc;
    API_CUDA(dcmt::stereo_entries_optimize_ig(entries_left, left_row_step_bytes, entries_right, right_row_step_bytes, elem_stride_bytes, disp,
                                              disp_pitch_bytes / sizeof(float), rows, cols, num_iterations, damp_factor, err_clip,
                                              static_cast<cudaStream_t>(cuda_stream)),
             "optimize_IG launch");
    return DCMT_OK;
}

int dcmt_get_initial_disparity_mat_f32(const float* depth, size_t depth_pitch_bytes, float* disp, size_t disp_pitch_bytes, int rows, int cols,
                                       float baseline, float focal, void* cuda_stream) {
    int rc = check_planes(rows, cols, 1);
    if (rc) return rc;
    if (rows > 65535) return fail(DCMT_E_UNSUPPORTED, "at most 65535 rows");
    if ((rc = check_mat_f32(depth, rows, cols, &depth_pitch_bytes)) || (rc = check_mat_f32(disp, rows, cols, &disp_pitch_bytes))) return rc;
    if ((rc = check_device())) return rc;
    API_CUDA(dcmt::stereo_initial_disparity_mat(depth, depth_pitch_bytes / sizeof(float), disp, disp_pitch_bytes / sizeof(float), rows, cols,
                                                baseline, focal, static_cast<cudaStream_t>(cuda_stream)),
             "initial disparity launch");
    return DCMT_OK;
}

int dcmt_retrieve_optimized_depth_mat_f32(const float* disp, size_t disp_pitch_bytes, float* depth, size_t depth_pitch_bytes, int rows, int cols,
                                          float baseline, float focal, float depth_clip, void* cuda_stream) {
    int rc = check_planes(rows, cols, 1);
    if (rc) return rc;
    if (rows > 65535) return fail(DCMT_E_UNSUPPORTED, "at most 65535 rows");
    if ((rc = check_mat_f32(disp, rows, cols, &disp_pitch_bytes)) || (rc = check_mat_f32(depth, rows, cols, &depth_pitch_bytes))) return rc;
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
    HostCall call;
    if ((rc = call.open(nullptr, 0, false))) return rc;
    cudaStream_t st = call.lanes[0].hs->s[0];
    const size_t used = (size_t)cols * elem_stride_bytes;
    Arena* ar = nullptr;
    if ((rc = arena_acquire(st, carve_bytes(used * rows, 1), &ar))) return rc;
    char* d = carve<char>(ar, used * rows);
    if ((rc = arena_ok(ar))) return rc;
    call.use(call.lanes[0]);
    API_CUDA(cudaMemcpy2DAsync(d, used, entries, row_step_bytes, used, rows, cudaMemcpyHostToDevice, st), "host to device copy");
    if ((rc = dcmt_entries_measurement_derivatives(d, rows, cols, used, elem_stride_bytes, st))) return rc;
    API_CUDA(cudaMemcpy2DAsync(entries, row_step_bytes, d, used, used, rows, cudaMemcpyDeviceToHost, st), "device to host copy");
    return call.finish();
}

int dcmt_entries_optimize_ig_host(const void* entries_left, size_t left_row_step_bytes, const void* entries_right,
                                  size_t right_row_step_bytes, size_t elem_stride_bytes, float* disp, size_t disp_pitch_bytes, int rows,
                                  int cols, int num_iterations, float damp_factor, float err_clip) {
    int rc = check_entries(entries_left, rows, cols, left_row_step_bytes, elem_stride_bytes);
    if (rc) return rc;
    if ((rc = check_entries(entries_right, rows, cols, right_row_step_bytes, elem_stride_bytes))) return rc;
    if ((rc = check_mat_f32(disp, rows, cols, &disp_pitch_bytes))) return rc;
    HostCall call;
    if ((rc = call.open(nullptr, 0, false))) return rc;
    cudaStream_t st = call.lanes[0].hs->s[0];
    const size_t used = (size_t)cols * elem_stride_bytes, drow = (size_t)cols * sizeof(float);
    Arena* ar = nullptr;
    if ((rc = arena_acquire(st, 2 * carve_bytes(used * rows, 1) + carve_bytes(drow * rows, 1), &ar))) return rc;
    char* dl = carve<char>(ar, used * rows);
    char* dr = carve<char>(ar, used * rows);
    float* dd = reinterpret_cast<float*>(carve<char>(ar, drow * rows));
    if ((rc = arena_ok(ar))) return rc;
    call.use(call.lanes[0]);
    API_CUDA(cudaMemcpy2DAsync(dl, used, entries_left, left_row_step_bytes, used, rows, cudaMemcpyHostToDevice, st), "host to device copy");
    API_CUDA(cudaMemcpy2DAsync(dr, used, entries_right, right_row_step_bytes, used, rows, cudaMemcpyHostToDevice, st), "host to device copy");
    API_CUDA(cudaMemcpy2DAsync(dd, drow, disp, disp_pitch_bytes, drow, rows, cudaMemcpyHostToDevice, st), "host to device copy");
    if ((rc = dcmt_entries_optimize_ig(dl, used, dr, used, elem_stride_bytes, dd, drow, rows, cols, num_iterations, damp_factor, err_clip, st)))
        return rc;
    API_CUDA(cudaMemcpy2DAsync(disp, disp_pitch_bytes, dd, drow, drow, rows, cudaMemcpyDeviceToHost, st), "device to host copy");
    return call.finish();
}

static int mat_pair_host(const float* in, size_t in_pitch, float* out, size_t out_pitch, int rows, int cols, int which, float baseline,
                         float focal, float clip) {
    int rc = check_planes(rows, cols, 1);
    if (rc) return rc;
    if ((rc = check_mat_f32(in, rows, cols, &in_pitch)) || (rc = check_mat_f32(out, rows, cols, &out_pitch))) return rc;
    HostCall call;
    if ((rc = call.open(nullptr, 0, false))) return rc;
    cudaStream_t st = call.lanes[0].hs->s[0];
    const size_t drow = (size_t)cols * sizeof(float);
    Arena* ar = nullptr;
    if ((rc = arena_acquire(st, 2 * carve_bytes(drow * rows, 1), &ar))) return rc;
    float* di = reinterpret_cast<float*>(carve<char>(ar, drow * rows));
    float* dout = reinterpret_cast<float*>(carve<char>(ar, drow * rows));
    if ((rc = arena_ok(ar))) return rc;
    call.use(call.lanes[0]);
    API_CUDA(cudaMemcpy2DAsync(di, drow, in, in_pitch, drow, rows, cudaMemcpyHostToDevice, st), "host to device copy");
    API_CUDA(cudaMemcpy2DAsync(dout, drow, out, out_pitch, drow, rows, cudaMemcpyHostToDevice, st), "host to device copy");  // untouched pixels keep their value
    rc = which == 0 ? dcmt_get_initial_disparity_mat_f32(di, drow, dout, drow, rows, cols, baseline, focal, st)
                    : dcmt_retrieve_optimized_depth_mat_f32(di, drow, dout, drow, rows, cols, baseline, focal, clip, st);
    if (rc) return rc;
    API_CUDA(cudaMemcpy2DAsync(out, out_pitch, dout, drow, drow, rows, cudaMemcpyDeviceToHost, st), "device to host copy");
    return call.finish();
}

int dcmt_get_initial_disparity_mat_f32_host(const float* depth, size_t depth_pitch_bytes, float* disp, size_t disp_pitch_bytes, int rows,
                                            int cols, float baseline, float focal) {
    return mat_pair_host(depth, depth_pitch_bytes, disp, disp_pitch_bytes, rows, cols, 0, baseline, focal, 0.0f);
}

int dcmt_retrieve_optimized_depth_mat_f32_host(const float* disp, size_t disp_pitch_bytes, float* depth, size_t depth_pitch_bytes, int rows,
                                               int cols, float baseline, float focal, float depth_clip) {
    return mat_pair_host(disp, disp_pitch_bytes, depth, depth_pitch_bytes, rows, cols, 1, baseline, focal, depth_clip);
}

}  // extern "C"
