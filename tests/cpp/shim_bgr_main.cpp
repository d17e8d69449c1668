// Test program for interpolate_with_superpixels_bgr / _bgr_to_u16 of include/img_completion.h: reads a raw CV_8UC3 BGR
// image and a raw CV_16UC1 depth image (metres * 256) and writes the float32 and uint16 results of the MatView overloads,
// every view with rows `pad` bytes longer than the image row (bytes past the row must stay untouched).  Compiled with the
// stand-in OpenCV headers of oracle/refshim it also makes the cv::Mat calls -- the BGR Mat with a padded step, as an ROI
// of a larger frame has -- writes their results and counts the type errors they throw.  Linked against the CPU emulator
// build by tests/test_superpixels_bgr.py, or against libdcmt.so on a GPU box.
//
//   shim_bgr ROWS COLS bgr.u8 in.u16 STEP NC OUT_PREFIX PAD  ->  OUT_PREFIX_view.{f32,u16} [, OUT_PREFIX_mat.{f32,u16}]
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

#include "img_completion.h"

static bool read_rows(const char* path, std::vector<uint8_t>& buf, int rows, size_t row, size_t step) {
    FILE* f = std::fopen(path, "rb");
    if (!f) return false;
    bool ok = true;
    for (int r = 0; r < rows && ok; ++r) ok = std::fread(buf.data() + r * step, 1, row, f) == row;
    std::fclose(f);
    return ok;
}

static bool write_rows(const std::string& path, const uint8_t* data, int rows, size_t row, size_t step, bool check_pad) {
    for (int r = 0; check_pad && r < rows; ++r)
        for (size_t i = row; i < step; ++i)
            if (data[r * step + i] != 0xA5) return false;
    FILE* f = std::fopen(path.c_str(), "wb");
    if (!f) return false;
    for (int r = 0; r < rows; ++r) std::fwrite(data + r * step, 1, row, f);
    std::fclose(f);
    return true;
}

int main(int argc, char** argv) {
    if (argc != 9) return 2;
    const int rows = std::atoi(argv[1]), cols = std::atoi(argv[2]), step = std::atoi(argv[5]), nc = std::atoi(argv[6]);
    const std::string out = argv[7];
    const size_t pad = (size_t)std::atoi(argv[8]);
    const size_t s3 = (size_t)cols * 3 + pad, s16 = (size_t)cols * 2 + pad, s32 = (size_t)cols * 4 + pad;
    std::vector<uint8_t> bgr((size_t)rows * s3, 0x5A), sparse((size_t)rows * s16, 0x5A);
    if (!read_rows(argv[3], bgr, rows, (size_t)cols * 3, s3) || !read_rows(argv[4], sparse, rows, (size_t)cols * 2, s16)) return 3;
    std::vector<uint8_t> o32((size_t)rows * s32, 0xA5), o16((size_t)rows * s16, 0xA5);
    dcmt::MatView vb{rows, cols, s3, bgr.data()}, vs{rows, cols, s16, sparse.data()};
    dcmt::MatView v32{rows, cols, s32, o32.data()}, v16{rows, cols, s16, o16.data()};
    try {
        // main_lc.cpp:182-220: cvtColor + generate_superpixels + interpolate_with_superpixels in one call
        dcmt::interpolate_with_superpixels_bgr(vb, vs, v32, step, nc);
        dcmt::interpolate_with_superpixels_bgr_to_u16(vb, vs, v16, step, nc);
    } catch (const std::exception& e) {
        std::fprintf(stderr, "%s\n", e.what());
        return 4;
    }
    if (!write_rows(out + "_view.f32", o32.data(), rows, (size_t)cols * 4, s32, true) ||
        !write_rows(out + "_view.u16", o16.data(), rows, (size_t)cols * 2, s16, true))
        return 5;
#ifdef DCMT_HAVE_OPENCV
    cv::Mat img(rows, cols, CV_8UC3, bgr.data());
    img.step = s3;  // an ROI's step: rows of a wider frame
    cv::Mat depth(rows, cols, CV_16UC1);
    for (int r = 0; r < rows; ++r) std::memcpy(depth.data + r * depth.step, sparse.data() + r * s16, (size_t)cols * 2);
    cv::Mat dense, dense16 = cv::Mat::zeros(3, 3, CV_8UC1);  // replaced by fresh matrices whatever they held
    try {
        dcmt::interpolate_with_superpixels_bgr(img, depth, dense, step, nc);
        dcmt::interpolate_with_superpixels_bgr_to_u16(img, depth, dense16, step, nc);
    } catch (const std::exception& e) {
        std::fprintf(stderr, "%s\n", e.what());
        return 6;
    }
    if (dense.type() != CV_32FC1 || dense16.type() != CV_16UC1 || !dense.isContinuous() || !dense16.isContinuous()) return 7;
    if (!write_rows(out + "_mat.f32", dense.data, rows, (size_t)cols * 4, dense.step, false) ||
        !write_rows(out + "_mat.u16", dense16.data, rows, (size_t)cols * 2, dense16.step, false))
        return 5;
    int thrown = 0;
    cv::Mat gray(rows, cols, CV_8UC1), depth32(rows, cols, CV_32FC1), scratch;
    try { dcmt::interpolate_with_superpixels_bgr(gray, depth, scratch, step, nc); } catch (const std::exception&) { ++thrown; }
    try { dcmt::interpolate_with_superpixels_bgr(img, depth32, scratch, step, nc); } catch (const std::exception&) { ++thrown; }
    try { dcmt::interpolate_with_superpixels_bgr_to_u16(depth, depth, scratch, step, nc); } catch (const std::exception&) { ++thrown; }
    std::printf("type errors thrown: %d\n", thrown);
#endif
    return 0;
}
