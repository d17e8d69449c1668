// Test program for dcmt::stereo_chain of include/img_completion.h: reads one Velodyne cloud, T and P (16 + 12 row-major floats)
// and a raw CV_8UC3 stereo pair, and writes the depth and disparity of the MatView overload, the BGR views with rows `pad`
// bytes longer than the image row (an ROI's step).  Compiled with the stand-in OpenCV headers of oracle/refshim it also makes
// the cv::Mat call, writes its results and counts the type and step errors it throws.  Linked against the CPU emulator build
// by tests/test_stereo_chain_call.py, or against libdcmt.so on a GPU box.
//
//   shim_chain ROWS COLS pts.f32 N_POINTS tp.f32 left.u8 right.u8 STEP NC OUT_PREFIX PAD
//     ->  OUT_PREFIX_view.{depth,disp} [, OUT_PREFIX_mat.{depth,disp}]
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

#include "img_completion.h"

static bool read_rows(const char* path, void* buf, int rows, size_t row, size_t step) {
    FILE* f = std::fopen(path, "rb");
    if (!f) return false;
    bool ok = true;
    for (int r = 0; r < rows && ok; ++r) ok = std::fread(static_cast<char*>(buf) + r * step, 1, row, f) == row;
    std::fclose(f);
    return ok;
}

static bool write_all(const std::string& path, const void* data, size_t bytes) {
    FILE* f = std::fopen(path.c_str(), "wb");
    if (!f) return false;
    const bool ok = std::fwrite(data, 1, bytes, f) == bytes;
    std::fclose(f);
    return ok;
}

int main(int argc, char** argv) {
    if (argc != 12) return 2;
    const int rows = std::atoi(argv[1]), cols = std::atoi(argv[2]), n_points = std::atoi(argv[4]), step = std::atoi(argv[8]);
    const int nc = std::atoi(argv[9]);
    const std::string out = argv[10];
    const size_t pad = (size_t)std::atoi(argv[11]), s3 = (size_t)cols * 3 + pad, plane = (size_t)rows * cols * 4;
    std::vector<float> pts((size_t)n_points * 4 + 1), tp(28);
    std::vector<uint8_t> left((size_t)rows * s3, 0x5A), right((size_t)rows * s3, 0x5A);
    if (!read_rows(argv[3], pts.data(), 1, (size_t)n_points * 16, 0) || !read_rows(argv[5], tp.data(), 1, 28 * 4, 0) ||
        !read_rows(argv[6], left.data(), rows, (size_t)cols * 3, s3) || !read_rows(argv[7], right.data(), rows, (size_t)cols * 3, s3))
        return 3;
    std::vector<float> depth((size_t)rows * cols, -7.0f), disp((size_t)rows * cols, -7.0f);
    dcmt::MatView vl{rows, cols, s3, left.data()}, vr{rows, cols, s3, right.data()};
    dcmt::MatView vd{rows, cols, (size_t)cols * 4, depth.data()}, vp{rows, cols, (size_t)cols * 4, disp.data()};
    try {
        dcmt::stereo_chain(pts.data(), n_points, tp.data(), tp.data() + 16, vl, vr, vd, step, nc, &vp);
    } catch (const std::exception& e) {
        std::fprintf(stderr, "%s\n", e.what());
        return 4;
    }
    if (!write_all(out + "_view.depth", depth.data(), plane) || !write_all(out + "_view.disp", disp.data(), plane)) return 5;
#ifdef DCMT_HAVE_OPENCV
    cv::Mat l(rows, cols, CV_8UC3, left.data()), r(rows, cols, CV_8UC3, right.data());
    l.step = s3;  // an ROI's step: rows of a wider frame
    r.step = s3;
    cv::Mat dm = cv::Mat::zeros(3, 3, CV_8UC1), pm;  // replaced by fresh matrices whatever they held
    try {
        dcmt::stereo_chain(pts.data(), n_points, tp.data(), tp.data() + 16, l, r, dm, step, nc, &pm);
    } catch (const std::exception& e) {
        std::fprintf(stderr, "%s\n", e.what());
        return 6;
    }
    if (dm.type() != CV_32FC1 || pm.type() != CV_32FC1 || !dm.isContinuous() || !pm.isContinuous()) return 7;
    if (!write_all(out + "_mat.depth", dm.data, plane) || !write_all(out + "_mat.disp", pm.data, plane)) return 5;
    int thrown = 0;
    cv::Mat gray(rows, cols, CV_8UC1), f32(rows, cols, CV_32FC1), packed(rows, cols, CV_8UC3), scratch;
    try { dcmt::stereo_chain(pts.data(), n_points, tp.data(), tp.data() + 16, gray, r, scratch, step, nc); } catch (const std::exception&) { ++thrown; }
    try { dcmt::stereo_chain(pts.data(), n_points, tp.data(), tp.data() + 16, l, f32, scratch, step, nc); } catch (const std::exception&) { ++thrown; }
    try { dcmt::stereo_chain(pts.data(), n_points, tp.data(), tp.data() + 16, l, packed, scratch, step, nc); } catch (const std::exception&) { ++thrown; }
    std::printf("type errors thrown: %d\n", thrown);
#endif
    return 0;
}
