// YUV 4:2:0 / 4:2:2 -> BGR arithmetic of cv2.cvtColor(frame, cv2.COLOR_YUV2BGR_<layout>), restated from OpenCV 4.13's
// imgproc/src/color_yuv.simd.hpp so that csrc/yuv.cu reproduces cv2 bit for bit.  Everything here is __host__ __device__: the
// kernel runs it in parallel, and tests/test_yuv_cpu.py compiles this header into a host library and compares it with cv2.
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

}  // namespace yuv
}  // namespace pn
