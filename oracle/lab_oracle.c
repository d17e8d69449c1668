/*
 * lab_oracle.c -- TEST INFRASTRUCTURE ONLY.  Plain-C CPU restatement of cv::cvtColor(COLOR_BGR2Lab) on 8-bit images,
 * the conversion the camera programs make in front of Slic::generate_superpixels (main_lc.cpp:182-183,
 * main_sl.cpp:438), with the semantics of OpenCV 4.13.0.  Checked against cv2 on all 2^24 colours and against a stored
 * sha256 of that result (tests/test_color_lab.py).
 *
 * Who may use it: tests/ and __graft_entry__.smoke() -- as the checker, never as the product.  The product (libdcmt.so)
 * does not link it.
 *
 * Build: oracle/lab_oracle.py  ->  oracle/liblab_oracle.so
 */
#include <math.h>
#include <stddef.h>
#include <stdint.h>

#define DCMT_ORACLE_API __attribute__((visibility("default")))
/* ---------------------------------------------------------------- cvtColor(COLOR_BGR2Lab), 8-bit
 * OpenCV 4.x RGB2Lab_b (modules/imgproc/src/color_lab.cpp) as called by main_lc.cpp:182-183 and main_sl.cpp:438: sRGB gamma
 * and the Lab cube root by table, XYZ with 12-bit and L, a, b with 15-bit fixed-point coefficients.  The tables are
 * restated here from their definition (the product's csrc/lab_tables.cuh is generated separately, by
 * oracle/make_lab_tables.py) with float / double in place of OpenCV's softfloat.  That reproduces every entry but one:
 * cube-root entry 324, 32768 * cbrt(324 / 2040) = 17745.4992 exactly, where the float-rounded cube root scales to exactly
 * 17745.5 and rounds half to even to 17746; OpenCV's softfloat cbrt is one ulp lower and its table holds 17745.
 * bgr, lab: rows x cols x 3 bytes, continuous. */
static uint16_t lab_gamma[256], lab_cbrt[2041];
static int lab_tables_ready;

static void lab_tables_init(void) {
    for (int v = 0; v < 256; ++v) {
        const double x = (float)v / 255.f;
        const double g = x <= 0.04045 ? x / 12.92 : pow((x + 0.055) / 1.055, 2.4);
        lab_gamma[v] = (uint16_t)lrintf(2040.f * (float)g); /* cvRound: half to even in the default rounding mode */
    }
    for (int i = 0; i < 2041; ++i) {
        const float x = (float)(1.0 / 2040) * (float)i;
        const float f = x < (float)(216.0 / 24389) ? x * (float)(841.0 / 108) + (float)(16.0 / 116) : (float)cbrt((double)x);
        lab_cbrt[i] = (uint16_t)lrintf(32768.f * f);
    }
    lab_cbrt[324] = 17745;
    lab_tables_ready = 1;
}

static inline int clamp255(int v) { return v < 0 ? 0 : (v > 255 ? 255 : v); }

DCMT_ORACLE_API void dcmt_oracle_bgr2lab(const uint8_t *bgr, uint8_t *lab, int rows, int cols) {
    if (!lab_tables_ready) lab_tables_init();
    for (size_t i = 0; i < (size_t)rows * cols; ++i) {
        const int B = lab_gamma[bgr[3 * i]], G = lab_gamma[bgr[3 * i + 1]], R = lab_gamma[bgr[3 * i + 2]];
        const int fX = lab_cbrt[(1777 * R + 1541 * G + 778 * B + 2048) >> 12];
        const int fY = lab_cbrt[(871 * R + 2929 * G + 296 * B + 2048) >> 12];
        const int fZ = lab_cbrt[(73 * R + 448 * G + 3575 * B + 2048) >> 12];
        lab[3 * i] = (uint8_t)clamp255((296 * fY - 1336934 + 16384) >> 15);
        lab[3 * i + 1] = (uint8_t)clamp255((500 * (fX - fY) + 128 * 32768 + 16384) >> 15);
        lab[3 * i + 2] = (uint8_t)clamp255((200 * (fY - fZ) + 128 * 32768 + 16384) >> 15);
    }
}
