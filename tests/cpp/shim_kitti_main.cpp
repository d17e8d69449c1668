// Test program for the KITTI uint16 functions of include/img_completion.h without OpenCV: reads a raw CV_16UC1 depth image
// (metres * 256) and a raw row-major int32 label map, and writes three raw results -- img_completion_u16_u16 (gaussian),
// interpolate_with_superpixels_u16 (float32) and interpolate_with_superpixels_u16_u16 -- each with rows `pad` bytes longer
// than the image row.  Linked against the CPU emulator build by tests/test_kitti_u16.py, or against libdcmt.so on a GPU box.
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

#define DCMT_NO_OPENCV 1
#include "img_completion.h"

template <class T>
static bool write_rows(const std::string& path, const std::vector<uint8_t>& buf, int rows, int cols, size_t step) {
    const size_t row = (size_t)cols * sizeof(T);
    for (int r = 0; r < rows; ++r)
        for (size_t i = row; i < step; ++i)
            if (buf[r * step + i] != 0xA5) return false;  // bytes past the row stay untouched
    FILE* f = std::fopen(path.c_str(), "wb");
    if (!f) return false;
    for (int r = 0; r < rows; ++r) std::fwrite(buf.data() + r * step, 1, row, f);
    std::fclose(f);
    return true;
}

int main(int argc, char** argv) {
    if (argc != 8) return 2;
    const int rows = std::atoi(argv[1]), cols = std::atoi(argv[2]), n_clusters = std::atoi(argv[5]), pad = std::atoi(argv[7]);
    const std::string out = argv[6];
    std::vector<uint16_t> in((size_t)rows * cols);
    std::vector<int32_t> lab((size_t)rows * cols);
    FILE* f = std::fopen(argv[3], "rb");
    if (!f || std::fread(in.data(), 2, in.size(), f) != in.size()) return 3;
    std::fclose(f);
    f = std::fopen(argv[4], "rb");
    if (!f || std::fread(lab.data(), 4, lab.size(), f) != lab.size()) return 3;
    std::fclose(f);
    std::vector<std::vector<int>> clusters(cols, std::vector<int>(rows));  // Slic::clusters is [col][row]
    for (int r = 0; r < rows; ++r)
        for (int c = 0; c < cols; ++c) clusters[c][r] = lab[(size_t)r * cols + c];
    const size_t step16 = (size_t)cols * 2 + pad, step32 = (size_t)cols * 4 + pad;
    std::vector<uint8_t> a1((size_t)rows * step16, 0xA5), a2f((size_t)rows * step32, 0xA5), a2u((size_t)rows * step16, 0xA5);
    dcmt::MatView sparse{rows, cols, (size_t)cols * 2, in.data()};
    dcmt::MatView v1{rows, cols, step16, a1.data()}, v2{rows, cols, step32, a2f.data()}, v3{rows, cols, step16, a2u.data()};
    try {
        dcmt::img_completion_u16_u16(sparse, v1, "gaussian");
        dcmt::interpolate_with_superpixels_u16(clusters, (size_t)n_clusters, sparse, v2, 1);
        dcmt::interpolate_with_superpixels_u16_u16(clusters, (size_t)n_clusters, sparse, v3, 1);
    } catch (const std::exception& e) {
        std::fprintf(stderr, "%s\n", e.what());
        return 4;
    }
    if (!write_rows<uint16_t>(out + "_a1.raw", a1, rows, cols, step16) || !write_rows<float>(out + "_a2.raw", a2f, rows, cols, step32) ||
        !write_rows<uint16_t>(out + "_a2u.raw", a2u, rows, cols, step16))
        return 5;
    return 0;
}
