// Test program for dcmt::bgr2lab of include/img_completion.h without OpenCV: reads a raw CV_8UC3 BGR image, converts it
// like main_lc.cpp:182-183 calls cv::cvtColor(img, lab, COLOR_BGR2Lab), with rows `pad` bytes longer than cols * 3 on
// both sides, and writes the Lab image (dense).  Linked against the CPU emulator build by tests/test_camera_chain_bgr.py,
// or against libdcmt.so on a GPU box.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#define DCMT_NO_OPENCV 1
#include "img_completion.h"

int main(int argc, char** argv) {
    if (argc != 6) return 2;
    const int rows = std::atoi(argv[1]), cols = std::atoi(argv[2]), pad = std::atoi(argv[5]);
    const size_t row = (size_t)cols * 3, step = row + pad;
    std::vector<uint8_t> in((size_t)rows * step, 0), out((size_t)rows * step, 7);
    FILE* f = std::fopen(argv[3], "rb");
    if (!f) return 3;
    for (int r = 0; r < rows; ++r)
        if (std::fread(in.data() + r * step, 1, row, f) != row) return 3;
    std::fclose(f);
    dcmt::MatView bgr{rows, cols, step, in.data()};
    dcmt::MatView lab{rows, cols, step, out.data()};
    try {
        dcmt::bgr2lab(bgr, lab);
    } catch (const std::exception& e) {
        std::fprintf(stderr, "%s\n", e.what());
        return 4;
    }
    for (int r = 0; r < rows; ++r)
        for (size_t i = row; i < step; ++i)
            if (out[r * step + i] != 7) return 5;  // bytes past cols * 3 stay untouched
    f = std::fopen(argv[4], "wb");
    for (int r = 0; r < rows; ++r) std::fwrite(out.data() + r * step, 1, row, f);
    std::fclose(f);
    return 0;
}
