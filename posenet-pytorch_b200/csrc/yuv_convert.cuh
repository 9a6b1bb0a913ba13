// YUV 4:2:0 / 4:2:2 -> BGR arithmetic of cv2.cvtColor(frame, cv2.COLOR_YUV2BGR_<layout>), restated from OpenCV 4.13's
// imgproc/src/color_yuv.simd.hpp so that csrc/yuv.cu reproduces cv2 bit for bit.  Everything here is __host__ __device__: the
// kernel runs it in parallel, and tests/test_yuv_cpu.py compiles this header into a host library and compares it with cv2.
// The inverse, BGR -> YUV (COLOR_BGR2YUV_<layout>, tests/test_yuv_out_cpu.py), follows `sample` at the end of the file.
//
//   BT.601 limited range in 20-bit fixed point, chroma nearest (a 2x2 block or a horizontal pair shares one U / V):
//     y = max(0, Y - 16) * 1220542,  u = U - 128,  v = V - 128
//     R = sat_u8((y + 1673527 v + 2^19) >> 20),  G = sat_u8((y - 852492 v - 409993 u + 2^19) >> 20),
//     B = sat_u8((y + 2116026 u + 2^19) >> 20)
#pragma once
#include <stdint.h>

#include "../../include/posenet_b200.h"

namespace pn {
namespace yuv {

constexpr int SHIFT = 20;
constexpr int CY = 1220542, CVR = 1673527, CVG = -852492, CUG = -409993, CUB = 2116026;

// The chroma terms of one U / V pair, shared by the pixels that sample it.
struct Chroma {
    int r, g, b;
};

__host__ __device__ inline Chroma chroma(int U, int V) {
    const int u = U - 128, v = V - 128, half = 1 << (SHIFT - 1);
    return {half + CVR * v, half + CVG * v + CUG * u, half + CUB * u};
}

__host__ __device__ inline uint8_t sat_u8(int x) { return (uint8_t)(x < 0 ? 0 : x > 255 ? 255 : x); }

// One pixel: bgr[0..2] = B, G, R.
__host__ __device__ inline void pixel(int Y, const Chroma &c, uint8_t *bgr) {
    const int y = (Y > 16 ? Y - 16 : 0) * CY;
    bgr[0] = sat_u8((y + c.b) >> SHIFT);
    bgr[1] = sat_u8((y + c.g) >> SHIFT);
    bgr[2] = sat_u8((y + c.r) >> SHIFT);
}

__host__ __device__ inline bool is_420(int layout) { return layout <= PN_YUV_NV21; }
__host__ __device__ inline bool is_planar(int layout) { return layout == PN_YUV_I420 || layout == PN_YUV_YV12; }

// Bytes of a frame of h x w (w even, h even for 4:2:0) in cv2's layout: [h * 3 / 2, w] for 4:2:0, [h, w, 2] for 4:2:2.
__host__ __device__ inline int64_t frame_bytes(int layout, int h, int w) {
    return is_420(layout) ? (int64_t)h * w * 3 / 2 : (int64_t)h * w * 2;
}

// The rows pixel row y samples: r0 is its luma row (4:2:0) or its packed row (4:2:2); r1 / r2 are the first / second chroma
// plane's rows (I420: U, V; YV12: V, U), r1 the interleaved chroma row (NV12 / NV21; r2 unused); both unused for 4:2:2.
__host__ __device__ inline void frame_rows(int layout, const uint8_t *f, int h, int w, int y, const uint8_t **r0,
                                           const uint8_t **r1, const uint8_t **r2) {
    const int64_t luma = (int64_t)h * w;
    if (!is_420(layout)) {
        *r0 = *r1 = *r2 = f + (int64_t)y * w * 2;
    } else if (is_planar(layout)) {
        *r0 = f + (int64_t)y * w;
        *r1 = f + luma + (int64_t)(y >> 1) * (w >> 1);
        *r2 = *r1 + luma / 4;
    } else {
        *r0 = f + (int64_t)y * w;
        *r1 = *r2 = f + luma + (int64_t)(y >> 1) * w;
    }
}

// Bytes of row r0 / r1 / r2 (which = 0, 1, 2) that hold n pixels (n even) from an even column on: 0 for a row the layout does
// not use.
__host__ __device__ inline int row_bytes(int layout, int which, int n) {
    if (which == 0) return is_420(layout) ? n : 2 * n;
    if (!is_420(layout)) return 0;
    if (is_planar(layout)) return n / 2;
    return which == 1 ? n : 0;
}

// The Y, U and V of pixel x of the row whose frame_rows are r0, r1, r2 (or of a copy of those rows that starts at an even
// column, with x counted from there).
__host__ __device__ inline void sample(int layout, const uint8_t *r0, const uint8_t *r1, const uint8_t *r2, int x, int *Y, int *U,
                                       int *V) {
    const int p = x & ~1;                      // the pair's first pixel
    switch (layout) {
    case PN_YUV_I420: *Y = r0[x]; *U = r1[x >> 1]; *V = r2[x >> 1]; break;
    case PN_YUV_YV12: *Y = r0[x]; *V = r1[x >> 1]; *U = r2[x >> 1]; break;
    case PN_YUV_NV12: *Y = r0[x]; *U = r1[p]; *V = r1[p + 1]; break;
    case PN_YUV_NV21: *Y = r0[x]; *V = r1[p]; *U = r1[p + 1]; break;
    case PN_YUV_YUY2: *Y = r0[2 * x]; *U = r0[2 * p + 1]; *V = r0[2 * p + 3]; break;
    case PN_YUV_UYVY: *Y = r0[2 * x + 1]; *U = r0[2 * p]; *V = r0[2 * p + 2]; break;
    default:          *Y = r0[2 * x]; *V = r0[2 * p + 1]; *U = r0[2 * p + 3]; break;   // PN_YUV_YVYU
    }
}

// ---- BGR -> YUV: cv2.cvtColor(frame, cv2.COLOR_BGR2YUV_<layout>), the output half (csrc/yuv.cu's bgr_to_yuv_kernel).  cv2
// runs two different arithmetic families, both BT.601 limited range:
//
//   4:2:0 (I420 / YV12), 20-bit fixed point; chroma is the top-left pixel's of each 2x2 block, the other three do not enter:
//     Y = (269484 R + 528482 G + 102760 B + 2^19 + (16 << 20)) >> 20
//     U = (-155188 R - 305135 G + 460324 B + 2^19 + (128 << 20)) >> 20,  V = (460324 R - 385875 G - 74448 B + ...) >> 20
//   4:2:2 (YUY2 / UYVY / YVYU), 14-bit fixed point; chroma is the pair's, from the sums sR, sG, sB of its two pixels (halved
//   coefficients, so an average):
//     Y = (4211 R + 8258 G + 1606 B + 2^13 + (16 << 14)) >> 14
//     U = (-1212 sR - 2384 sG + 3596 sB + 2^13 + (128 << 14)) >> 14,  V = (3596 sR - 3015 sG - 582 sB + ...) >> 14
//
// None of these leaves 16..240 for uint8 input; the saturation is kept so the functions hold for any int input.
constexpr int CRY = 269484, CGY = 528482, CBY = 102760, CRU = -155188, CGU = -305135, CBU = 460324, CGV = -385875, CBV = -74448;
constexpr int SHIFT422 = 14;
constexpr int R2Y422 = 4211, G2Y422 = 8258, B2Y422 = 1606, R2U422 = -1212, G2U422 = -2384, B2U422 = 3596, R2V422 = 3596,
              G2V422 = -3015, B2V422 = -582;

__host__ __device__ inline uint8_t luma_420(int b, int g, int r) {
    return sat_u8((CRY * r + CGY * g + CBY * b + (1 << (SHIFT - 1)) + (16 << SHIFT)) >> SHIFT);
}

__host__ __device__ inline void chroma_420(int b, int g, int r, uint8_t *U, uint8_t *V) {
    const int c = (1 << (SHIFT - 1)) + (128 << SHIFT);
    *U = sat_u8((CRU * r + CGU * g + CBU * b + c) >> SHIFT);
    *V = sat_u8((CBU * r + CGV * g + CBV * b + c) >> SHIFT);
}

__host__ __device__ inline uint8_t luma_422(int b, int g, int r) {
    return sat_u8((R2Y422 * r + G2Y422 * g + B2Y422 * b + (1 << (SHIFT422 - 1)) + (16 << SHIFT422)) >> SHIFT422);
}

// sb, sg, sr: the sums of the pair's two pixels (0..510).
__host__ __device__ inline void chroma_422(int sb, int sg, int sr, uint8_t *U, uint8_t *V) {
    const int c = (1 << (SHIFT422 - 1)) + (128 << SHIFT422);
    *U = sat_u8((R2U422 * sr + G2U422 * sg + B2U422 * sb + c) >> SHIFT422);
    *V = sat_u8((R2V422 * sr + G2V422 * sg + B2V422 * sb + c) >> SHIFT422);
}

// Converts pixels x, x + 1 (x even) of BGR row `bgr` and stores them in the rows r0, r1, r2 of frame_rows (or in copies of
// them that start at an even column, x counted from there): both lumas, and the pair's U and V where the row carries chroma --
// every row of 4:2:2, the even rows of 4:2:0.  The inverse of `sample`, for the five layouts cv2 writes (not NV12 / NV21).
__host__ __device__ inline void put_pair(int layout, const uint8_t *bgr, int x, bool even_row, uint8_t *r0, uint8_t *r1,
                                         uint8_t *r2) {
    const uint8_t *p = bgr + 3 * x;
    if (is_420(layout)) {
        r0[x] = luma_420(p[0], p[1], p[2]);
        r0[x + 1] = luma_420(p[3], p[4], p[5]);
        if (even_row) {
            uint8_t U, V;
            chroma_420(p[0], p[1], p[2], &U, &V);
            (layout == PN_YUV_I420 ? r1 : r2)[x >> 1] = U;
            (layout == PN_YUV_I420 ? r2 : r1)[x >> 1] = V;
        }
        return;
    }
    const uint8_t Y0 = luma_422(p[0], p[1], p[2]), Y1 = luma_422(p[3], p[4], p[5]);
    uint8_t U, V;
    chroma_422(p[0] + p[3], p[1] + p[4], p[2] + p[5], &U, &V);
    uint8_t *q = r0 + 2 * x;
    switch (layout) {
    case PN_YUV_YUY2: q[0] = Y0; q[1] = U; q[2] = Y1; q[3] = V; break;
    case PN_YUV_UYVY: q[0] = U; q[1] = Y0; q[2] = V; q[3] = Y1; break;
    default:          q[0] = Y0; q[1] = V; q[2] = Y1; q[3] = U; break;     // PN_YUV_YVYU
    }
}

}  // namespace yuv
}  // namespace pn
