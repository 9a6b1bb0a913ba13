// Rasteriser arithmetic of posenet.utils.draw_skel_and_kp (cv2.drawKeypoints with DRAW_RICH_KEYPOINTS, then cv2.polylines),
// restated from OpenCV's imgproc/src/drawing.cpp and features2d/src/draw.cpp so that csrc/draw.cu reproduces cv2 bit for bit.
// Everything here is __host__ __device__: the kernel runs it in parallel, and tests/test_draw_cpu.py compiles this header into
// a host library and compares it with cv2.
//
//   keypoint k -> circle(center = cvRound(x * 16), radius = cvRound(size / 2 * 16), LINE_AA, shift 4)
//              -> EllipseEx: ellipse2Poly (double, SinTable) -> points rounded into 16.16 fixed point -> LineAA per pair
//   segment    -> Line (LINE_8, LineIterator with connectivity 8; clipLine only when an endpoint is off the frame)
//
// LineAA pixel order inside one call does not matter (each major-axis step touches its own column / row), but the blends of
// different calls that land on one pixel must run in cv2's order.  Each LineAA put blends every channel TWICE with the same
// alpha (the 3-channel ICV_PUT_POINT of drawing.cpp).
#pragma once
#include <math.h>
#include <stdint.h>

namespace pn {
namespace raster {

constexpr int XY_SHIFT = 16;
constexpr int64_t XY_ONE = int64_t(1) << XY_SHIFT;
constexpr int DRAW_SHIFT = 4;                  // features2d draw.cpp: draw_shift_bits (draw_multiplier = 16)

// The three tables of OpenCV's imgproc/src/drawing.cpp (Apache-2.0), read from the cv2 4.13 binary: SinTable float[451]
// (sin of whole degrees 0..450), FilterTable int[64] (the LineAA footprint weights), SlopeCorrTable uchar[32].
#define PN_RASTER_SIN_TABLE {                                                                                          \
    0.f, 0.0174524002f, 0.0348994993f, 0.0523359999f, 0.0697565004f, 0.0871556997f, 0.104528502f, 0.121869303f, \
    0.139173105f, 0.156434506f, 0.173648193f, 0.190808997f, 0.2079117f, 0.224951103f, 0.241921902f, 0.258819014f, \
    0.275637388f, 0.29237169f, 0.309017003f, 0.325568199f, 0.342020094f, 0.35836789f, 0.374606609f, 0.390731096f, \
    0.406736612f, 0.4226183f, 0.438371092f, 0.453990489f, 0.469471604f, 0.484809607f, 0.5f, 0.515038073f, \
    0.529919326f, 0.544638991f, 0.559192896f, 0.573576391f, 0.587785304f, 0.601814985f, 0.615661502f, 0.629320383f, \
    0.642787576f, 0.656059027f, 0.669130623f, 0.681998372f, 0.694658399f, 0.707106829f, 0.719339788f, 0.7313537f, \
    0.74314481f, 0.754709601f, 0.766044378f, 0.777145982f, 0.788010776f, 0.798635483f, 0.809017003f, 0.819151998f, \
    0.829037607f, 0.838670611f, 0.848048091f, 0.857167304f, 0.866025388f, 0.874619722f, 0.882947624f, 0.891006529f, \
    0.898793995f, 0.906307817f, 0.913545489f, 0.920504928f, 0.927183926f, 0.933580399f, 0.939692616f, 0.945518613f, \
    0.95105648f, 0.956304789f, 0.96126169f, 0.965925813f, 0.970295727f, 0.974370122f, 0.978147626f, 0.981627226f, \
    0.984807789f, 0.987688303f, 0.990268111f, 0.992546201f, 0.994521916f, 0.99619472f, 0.997564077f, 0.99862951f, \
    0.999390781f, 0.99984771f, 1.f, 0.99984771f, 0.999390781f, 0.99862951f, 0.997564077f, 0.99619472f, \
    0.994521916f, 0.992546201f, 0.990268111f, 0.987688303f, 0.984807789f, 0.981627226f, 0.978147626f, 0.974370122f, \
    0.970295727f, 0.965925813f, 0.96126169f, 0.956304789f, 0.95105648f, 0.945518613f, 0.939692616f, 0.933580399f, \
    0.927183926f, 0.920504928f, 0.913545489f, 0.906307817f, 0.898793995f, 0.891006529f, 0.882947624f, 0.874619722f, \
    0.866025388f, 0.857167304f, 0.848048091f, 0.838670611f, 0.829037607f, 0.819151998f, 0.809017003f, 0.798635483f, \
    0.788010776f, 0.777145982f, 0.766044378f, 0.754709601f, 0.74314481f, 0.7313537f, 0.719339788f, 0.707106829f, \
    0.694658399f, 0.681998372f, 0.669130623f, 0.656059027f, 0.642787576f, 0.629320383f, 0.615661502f, 0.601814985f, \
    0.587785304f, 0.573576391f, 0.559192896f, 0.544638991f, 0.529919326f, 0.515038073f, 0.5f, 0.484809607f, \
    0.469471604f, 0.453990489f, 0.438371092f, 0.4226183f, 0.406736612f, 0.390731096f, 0.374606609f, 0.35836789f, \
    0.342020094f, 0.325568199f, 0.309017003f, 0.29237169f, 0.275637388f, 0.258819014f, 0.241921902f, 0.224951103f, \
    0.2079117f, 0.190808997f, 0.173648193f, 0.156434506f, 0.139173105f, 0.121869303f, 0.104528502f, 0.0871556997f, \
    0.0697565004f, 0.0523359999f, 0.0348994993f, 0.0174524002f, 0.f, -0.0174524002f, -0.0348994993f, -0.0523359999f, \
    -0.0697565004f, -0.0871556997f, -0.104528502f, -0.121869303f, -0.139173105f, -0.156434506f, -0.173648193f, -0.190808997f, \
    -0.2079117f, -0.224951103f, -0.241921902f, -0.258819014f, -0.275637388f, -0.29237169f, -0.309017003f, -0.325568199f, \
    -0.342020094f, -0.35836789f, -0.374606609f, -0.390731096f, -0.406736612f, -0.4226183f, -0.438371092f, -0.453990489f, \
    -0.469471604f, -0.484809607f, -0.5f, -0.515038073f, -0.529919326f, -0.544638991f, -0.559192896f, -0.573576391f, \
    -0.587785304f, -0.601814985f, -0.615661502f, -0.629320383f, -0.642787576f, -0.656059027f, -0.669130623f, -0.681998372f, \
    -0.694658399f, -0.707106829f, -0.719339788f, -0.7313537f, -0.74314481f, -0.754709601f, -0.766044378f, -0.777145982f, \
    -0.788010776f, -0.798635483f, -0.809017003f, -0.819151998f, -0.829037607f, -0.838670611f, -0.848048091f, -0.857167304f, \
    -0.866025388f, -0.874619722f, -0.882947624f, -0.891006529f, -0.898793995f, -0.906307817f, -0.913545489f, -0.920504928f, \
    -0.927183926f, -0.933580399f, -0.939692616f, -0.945518613f, -0.95105648f, -0.956304789f, -0.96126169f, -0.965925813f, \
    -0.970295727f, -0.974370122f, -0.978147626f, -0.981627226f, -0.984807789f, -0.987688303f, -0.990268111f, -0.992546201f, \
    -0.994521916f, -0.99619472f, -0.997564077f, -0.99862951f, -0.999390781f, -0.99984771f, -1.f, -0.99984771f, \
    -0.999390781f, -0.99862951f, -0.997564077f, -0.99619472f, -0.994521916f, -0.992546201f, -0.990268111f, -0.987688303f, \
    -0.984807789f, -0.981627226f, -0.978147626f, -0.974370122f, -0.970295727f, -0.965925813f, -0.96126169f, -0.956304789f, \
    -0.95105648f, -0.945518613f, -0.939692616f, -0.933580399f, -0.927183926f, -0.920504928f, -0.913545489f, -0.906307817f, \
    -0.898793995f, -0.891006529f, -0.882947624f, -0.874619722f, -0.866025388f, -0.857167304f, -0.848048091f, -0.838670611f, \
    -0.829037607f, -0.819151998f, -0.809017003f, -0.798635483f, -0.788010776f, -0.777145982f, -0.766044378f, -0.754709601f, \
    -0.74314481f, -0.7313537f, -0.719339788f, -0.707106829f, -0.694658399f, -0.681998372f, -0.669130623f, -0.656059027f, \
    -0.642787576f, -0.629320383f, -0.615661502f, -0.601814985f, -0.587785304f, -0.573576391f, -0.559192896f, -0.544638991f, \
    -0.529919326f, -0.515038073f, -0.5f, -0.484809607f, -0.469471604f, -0.453990489f, -0.438371092f, -0.4226183f, \
    -0.406736612f, -0.390731096f, -0.374606609f, -0.35836789f, -0.342020094f, -0.325568199f, -0.309017003f, -0.29237169f, \
    -0.275637388f, -0.258819014f, -0.241921902f, -0.224951103f, -0.2079117f, -0.190808997f, -0.173648193f, -0.156434506f, \
    -0.139173105f, -0.121869303f, -0.104528502f, -0.0871556997f, -0.0697565004f, -0.0523359999f, -0.0348994993f, -0.0174524002f, \
    -0.f, 0.0174524002f, 0.0348994993f, 0.0523359999f, 0.0697565004f, 0.0871556997f, 0.104528502f, 0.121869303f, \
    0.139173105f, 0.156434506f, 0.173648193f, 0.190808997f, 0.2079117f, 0.224951103f, 0.241921902f, 0.258819014f, \
    0.275637388f, 0.29237169f, 0.309017003f, 0.325568199f, 0.342020094f, 0.35836789f, 0.374606609f, 0.390731096f, \
    0.406736612f, 0.4226183f, 0.438371092f, 0.453990489f, 0.469471604f, 0.484809607f, 0.5f, 0.515038073f, \
    0.529919326f, 0.544638991f, 0.559192896f, 0.573576391f, 0.587785304f, 0.601814985f, 0.615661502f, 0.629320383f, \
    0.642787576f, 0.656059027f, 0.669130623f, 0.681998372f, 0.694658399f, 0.707106829f, 0.719339788f, 0.7313537f, \
    0.74314481f, 0.754709601f, 0.766044378f, 0.777145982f, 0.788010776f, 0.798635483f, 0.809017003f, 0.819151998f, \
    0.829037607f, 0.838670611f, 0.848048091f, 0.857167304f, 0.866025388f, 0.874619722f, 0.882947624f, 0.891006529f, \
    0.898793995f, 0.906307817f, 0.913545489f, 0.920504928f, 0.927183926f, 0.933580399f, 0.939692616f, 0.945518613f, \
    0.95105648f, 0.956304789f, 0.96126169f, 0.965925813f, 0.970295727f, 0.974370122f, 0.978147626f, 0.981627226f, \
    0.984807789f, 0.987688303f, 0.990268111f, 0.992546201f, 0.994521916f, 0.99619472f, 0.997564077f, 0.99862951f, \
    0.999390781f, 0.99984771f, 1.f \
    }
#define PN_RASTER_FILTER_TABLE {                                                                                       \
    168, 177, 185, 194, 202, 210, 218, 224, 231, 236, 241, 246, 249, 252, 254, 254,                                    \
    254, 254, 252, 249, 246, 241, 236, 231, 224, 218, 210, 202, 194, 185, 177, 168,                                    \
    158, 149, 140, 131, 122, 114, 105, 97, 89, 82, 75, 68, 62, 56, 50, 45,                                             \
    40, 36, 32, 28, 25, 22, 19, 16, 14, 12, 11, 9, 8, 7, 5, 5 }
#define PN_RASTER_SLOPE_CORR_TABLE {                                                                                   \
    181, 181, 181, 182, 182, 183, 184, 185, 187, 188, 190, 192, 194, 196, 198, 201,                                    \
    203, 206, 209, 211, 214, 218, 221, 224, 227, 231, 235, 238, 242, 246, 250, 254 }

#ifdef __CUDACC__
__device__ const float kSinTableDev[451] = PN_RASTER_SIN_TABLE;
__device__ const int kFilterTableDev[64] = PN_RASTER_FILTER_TABLE;
__device__ const uint8_t kSlopeCorrTableDev[32] = PN_RASTER_SLOPE_CORR_TABLE;
#define PN_HD __host__ __device__ __forceinline__
#else
#define PN_HD inline
#endif
static const float kSinTableHost[451] = PN_RASTER_SIN_TABLE;
static const int kFilterTableHost[64] = PN_RASTER_FILTER_TABLE;
static const uint8_t kSlopeCorrTableHost[32] = PN_RASTER_SLOPE_CORR_TABLE;

PN_HD float sin_table(int i) {
#ifdef __CUDA_ARCH__
    return kSinTableDev[i];
#else
    return kSinTableHost[i];
#endif
}
PN_HD int filter_table(int i) {
#ifdef __CUDA_ARCH__
    return kFilterTableDev[i];
#else
    return kFilterTableHost[i];
#endif
}
PN_HD int slope_corr_table(int i) {
#ifdef __CUDA_ARCH__
    return kSlopeCorrTableDev[i];
#else
    return kSlopeCorrTableHost[i];
#endif
}

// Unfused IEEE double arithmetic (ellipse2Poly and clipLine must not contract into FMAs).
PN_HD double dmul(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
PN_HD double dadd(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}
PN_HD double ddiv(double a, double b) {
#ifdef __CUDA_ARCH__
    return __ddiv_rn(a, b);
#else
    return a / b;
#endif
}

// cvRound (round half to even); a result outside int32 (or NaN) gives INT_MIN, what the x86 conversion cv2 uses returns.
// posenet.constants.CONNECTED_PART_INDICES: the limbs draw_skeleton connects, in list order.
constexpr int NUM_LIMBS = 12;
#define PN_RASTER_LIMBS {11, 5, 7, 5, 7, 9, 11, 13, 13, 15, 12, 6, 8, 6, 8, 10, 12, 14, 14, 16, 5, 6, 11, 12}
#ifdef __CUDACC__
__device__ const uint8_t kLimbsDev[2 * NUM_LIMBS] = PN_RASTER_LIMBS;
#endif
static const uint8_t kLimbsHost[2 * NUM_LIMBS] = PN_RASTER_LIMBS;
PN_HD int limb_part(int limb, int end) {
#ifdef __CUDA_ARCH__
    return kLimbsDev[2 * limb + end];
#else
    return kLimbsHost[2 * limb + end];
#endif
}

// Pose selection.  draw_skel_and_kp skips a pose when `score < min_pose_score`; draw_skeleton keeps it when
// `score >= min_pose_confidence` (the two differ for a NaN score only).
PN_HD bool pose_selected(double score, double min_pose, bool with_keypoints) {
    return with_keypoints ? !(score < min_pose) : score >= min_pose;
}

PN_HD int cv_round(double v) {
    const double r = rint(v);
    return (r >= -2147483648.0 && r < 2147483648.0) ? (int)r : INT32_MIN;
}
PN_HD int cv_round(float v) {
    const float r = rintf(v);
    return (r >= -2147483648.f && r < 2147483648.f) ? (int)r : INT32_MIN;
}
// numpy's astype(np.int32) of a float64: truncation toward zero, INT_MIN outside int32 (or NaN).
PN_HD int trunc_i32(double v) { return (v > -2147483649.0 && v < 2147483648.0) ? (int)v : INT32_MIN; }

// ---- selection (posenet/utils.py: _keypoints_above / get_adjacent_keypoints) -----------------------------------------
// A keypoint is cv2.KeyPoint(float(x), float(y), 10. * float(score)): float32 fields, the size product taken in float64.
// drawKeypoints turns it into a circle in 1/16 px (draw_shift_bits = 4).
struct Circle {
    int cx, cy, r;                             // 1/16 px, as _drawKeypoint passes them to cv::circle
};
PN_HD Circle keypoint_circle(double y, double x, double score) {
    const float xf = (float)x, yf = (float)y, sf = (float)dmul(10.0, score);
    Circle c;
    c.cx = cv_round(xf * 16.f);
    c.cy = cv_round(yf * 16.f);
    c.r = cv_round(sf / 2.f * 16.f);
    return c;
}

// ---- EllipseEx / ellipse2Poly for a full circle (angle 0, arc 0..360) ---------------------------------------------------
struct Poly {
    int64_t cx, cy, r;                         // 16.16 fixed point (circle() shifts by XY_SHIFT - shift)
    int delta, npts;                           // ellipse2Poly step in degrees and point count (0, delta, .., 360)
};
PN_HD Poly circle_poly(const Circle &c) {
    Poly p;
    p.cx = (int64_t)c.cx << (XY_SHIFT - DRAW_SHIFT);
    p.cy = (int64_t)c.cy << (XY_SHIFT - DRAW_SHIFT);
    const int64_t r = (int64_t)c.r << (XY_SHIFT - DRAW_SHIFT);
    p.r = r < 0 ? -r : r;                      // EllipseEx takes |axes|
    const int d = (int)((p.r + (XY_ONE >> 1)) >> XY_SHIFT);
    p.delta = d < 3 ? 90 : d < 10 ? 30 : d < 15 ? 18 : 5;
    p.npts = 360 / p.delta + 1;
    return p;
}
// Point k of the polygon, rounded as EllipseEx does: cvRound(v / XY_ONE) << XY_SHIFT, plus cvRound of the remainder.
// With angle 0, ellipse2Poly's rotation is alpha = 1, beta = 0, so cx + x*alpha - y*beta is exactly cx + x (and cy + y).
PN_HD void poly_point(const Poly &p, int k, int64_t *px, int64_t *py) {
    const int a = k * p.delta;                 // every delta divides 360: no clamping to arc_end
    const double x = dmul((double)p.r, (double)sin_table(450 - a));
    const double y = dmul((double)p.r, (double)sin_table(a));
    const double vx = dadd((double)p.cx, x), vy = dadd((double)p.cy, y);
    int64_t X = (int64_t)cv_round(vx / (double)XY_ONE) << XY_SHIFT;
    int64_t Y = (int64_t)cv_round(vy / (double)XY_ONE) << XY_SHIFT;
    X += cv_round(dadd(vx, -(double)X));
    Y += cv_round(dadd(vy, -(double)Y));
    *px = X;
    *py = Y;
}

// ---- clipLine (drawing.cpp, int64 form; both LineAA and LineIterator use it) ----------------------------------------
PN_HD bool clip_line(int64_t w, int64_t h, int64_t &x1, int64_t &y1, int64_t &x2, int64_t &y2) {
    if (w <= 0 || h <= 0) return false;
    const int64_t right = w - 1, bottom = h - 1;
    int c1 = (x1 < 0) + (x1 > right) * 2 + (y1 < 0) * 4 + (y1 > bottom) * 8;
    int c2 = (x2 < 0) + (x2 > right) * 2 + (y2 < 0) * 4 + (y2 > bottom) * 8;
    if ((c1 & c2) == 0 && (c1 | c2) != 0) {
        int64_t a;
        if (c1 & 12) {
            a = c1 < 8 ? 0 : bottom;
            x1 += (int64_t)ddiv(dmul((double)(a - y1), (double)(x2 - x1)), (double)(y2 - y1));
            y1 = a;
            c1 = (x1 < 0) + (x1 > right) * 2;
        }
        if (c2 & 12) {
            a = c2 < 8 ? 0 : bottom;
            x2 += (int64_t)ddiv(dmul((double)(a - y2), (double)(x2 - x1)), (double)(y2 - y1));
            y2 = a;
            c2 = (x2 < 0) + (x2 > right) * 2;
        }
        if ((c1 & c2) == 0 && (c1 | c2) != 0) {
            if (c1) {
                a = c1 == 1 ? 0 : right;
                y1 += (int64_t)ddiv(dmul((double)(a - x1), (double)(y2 - y1)), (double)(x2 - x1));
                x1 = a;
                c1 = 0;
            }
            if (c2) {
                a = c2 == 1 ? 0 : right;
                y2 += (int64_t)ddiv(dmul((double)(a - x2), (double)(y2 - y1)), (double)(x2 - x1));
                x2 = a;
                c2 = 0;
            }
        }
    }
    return (c1 | c2) == 0;
}

// ---- LineAA (drawing.cpp) split into a setup and an independent step function -----------------------------------------
// Step s = 0 .. ecount is one iteration of cv2's loop: the pixel column (x_major) or row at `start + s`, three puts across it.
struct LineAA {
    int64_t p1;                                // minor-axis coordinate of step 0 (16.16, +1/2 and end-point adjusted)
    int64_t inc;                               // its increment per step (y_step or x_step)
    int start, ecount;                         // major-axis pixel of step 0; last step index
    bool x_major;
    int ep[9];                                 // end-point correction table
};
PN_HD bool lineaa_setup(int w, int h, int64_t x1, int64_t y1, int64_t x2, int64_t y2, LineAA &L) {
    if (!clip_line((int64_t)w << XY_SHIFT, (int64_t)h << XY_SHIFT, x1, y1, x2, y2)) return false;
    int64_t dx = x2 - x1, dy = y2 - y1;
    int64_t j = dx < 0 ? -1 : 0;
    const int64_t ax = (dx ^ j) - j;
    int64_t i = dy < 0 ? -1 : 0;
    const int64_t ay = (dy ^ i) - i;
    int slope;
    if (ax > ay) {
        dy = (dy ^ j) - j;
        if (j) { int64_t t = x1; x1 = x2; x2 = t; t = y1; y1 = y2; y2 = t; }
        const int64_t ys = (dy << XY_SHIFT) / (ax | 1);
        x2 += XY_ONE;
        L.ecount = (int)((x2 >> XY_SHIFT) - (x1 >> XY_SHIFT));
        j = -(x1 & (XY_ONE - 1));
        L.p1 = y1 + ((ys * j) >> XY_SHIFT) + (XY_ONE >> 1);
        L.inc = ys;
        slope = (int)((ys >> (XY_SHIFT - 5)) & 0x3f);
        slope ^= (ys < 0 ? 0x3f : 0);
        i = (x1 >> (XY_SHIFT - 7)) & 0x78;
        j = (x2 >> (XY_SHIFT - 7)) & 0x78;
        L.start = (int)(x1 >> XY_SHIFT);
        L.x_major = true;
    } else {
        dx = (dx ^ i) - i;
        if (i) { int64_t t = x1; x1 = x2; x2 = t; t = y1; y1 = y2; y2 = t; }
        const int64_t xs = (dx << XY_SHIFT) / (ay | 1);
        y2 += XY_ONE;
        L.ecount = (int)((y2 >> XY_SHIFT) - (y1 >> XY_SHIFT));
        j = -(y1 & (XY_ONE - 1));
        L.p1 = x1 + ((xs * j) >> XY_SHIFT) + (XY_ONE >> 1);
        L.inc = xs;
        slope = (int)((xs >> (XY_SHIFT - 5)) & 0x3f);
        slope ^= (xs < 0 ? 0x3f : 0);
        i = (y1 >> (XY_SHIFT - 7)) & 0x78;
        j = (y2 >> (XY_SHIFT - 7)) & 0x78;
        L.start = (int)(y1 >> XY_SHIFT);
        L.x_major = false;
    }
    slope = (slope & 0x20) ? 0x100 : slope_corr_table(slope);
    const int t0 = slope << 7;
    const int t1 = ((0x78 - (int)i) | 4) * slope;
    const int t2 = ((int)j | 4) * slope;
    L.ep[0] = 0;
    L.ep[8] = slope;
    L.ep[1] = L.ep[3] = ((((int)(j - i) & 0x78) | 4) * slope >> 8) & 0x1ff;
    L.ep[2] = (t1 >> 8) & 0x1ff;
    L.ep[4] = ((((int)(j - i) + 0x80) | 4) * slope >> 8) & 0x1ff;
    L.ep[5] = ((t1 + t0) >> 8) & 0x1ff;
    L.ep[6] = (t2 >> 8) & 0x1ff;
    L.ep[7] = ((t2 + t0) >> 8) & 0x1ff;
    return true;
}
// Step s: the major-axis pixel, the minor-axis pixel of the first of the three puts (the others follow at +1, +2) and their
// alphas.  The caller bounds-checks each put, as cv2 does.
PN_HD void lineaa_step(const LineAA &L, int s, int *major, int *minor0, int alpha[3]) {
    const int e = L.ecount - s;
    const int64_t m = L.p1 + (int64_t)s * L.inc;   // cv2 adds inc once per step; the product is the same int64
    *major = L.start + s;
    *minor0 = (int)((m >> XY_SHIFT) - 1);
    const int ep = L.ep[(((s >= 2) + 1) & (s | 2)) * 3 + (((e >= 2) + 1) & (e | 2))];
    const int dist = (int)((m >> (XY_SHIFT - 5)) & 31);
    alpha[0] = (ep * filter_table(dist + 32) >> 8) & 0xff;
    alpha[1] = (ep * filter_table(dist) >> 8) & 0xff;
    alpha[2] = (ep * filter_table(63 - dist) >> 8) & 0xff;
}
// ICV_PUT_POINT for 3 channels: two blends with the same alpha.
PN_HD void blend_put(uint8_t *px, const uint8_t col[3], int a) {
    for (int c = 0; c < 3; ++c) {
        int v = px[c];
        v += ((col[c] - v) * a + 127) >> 8;
        v += ((col[c] - v) * a + 127) >> 8;
        px[c] = (uint8_t)v;
    }
}

// ---- Line with LINE_8 (LineIterator, connectivity 8, left to right) ---------------------------------------------------
// Pixel i of the iterator in closed form: after i steps the Bresenham error has taken k_i = floor((2dy*i + dx - 1) / 2dx)
// "plus" steps (err = dx - 2dy, plusDelta = 2dx, minusDelta = -2dy), so the pixels can be produced in any order.
struct Line8 {
    int x1, y1, dx, dy, sx, sy, count;
    bool vert;
};
PN_HD bool line8_setup(int w, int h, int x1, int y1, int x2, int y2, Line8 &L) {
    if ((unsigned)x1 >= (unsigned)w || (unsigned)x2 >= (unsigned)w || (unsigned)y1 >= (unsigned)h || (unsigned)y2 >= (unsigned)h) {
        int64_t a = x1, b = y1, c = x2, d = y2;
        if (!clip_line(w, h, a, b, c, d)) return false;
        x1 = (int)a; y1 = (int)b; x2 = (int)c; y2 = (int)d;
    }
    int dx = x2 - x1, dy = y2 - y1, sx = 1, sy = 1;
    if (dx < 0) {
        dx = -dx; dy = -dy;
        int t = x1; x1 = x2; x2 = t;
        t = y1; y1 = y2; y2 = t;
    }
    if (dy < 0) { dy = -dy; sy = -1; }
    L.vert = dy > dx;
    if (L.vert) { int t = dx; dx = dy; dy = t; t = sx; sx = sy; sy = t; }
    L.x1 = x1; L.y1 = y1; L.dx = dx; L.dy = dy; L.sx = sx; L.sy = sy;
    L.count = dx + 1;
    return true;
}
PN_HD void line8_pixel(const Line8 &L, int i, int *x, int *y) {
    const int k = L.dx ? (int)((2 * (int64_t)L.dy * i + L.dx - 1) / (2 * (int64_t)L.dx)) : 0;
    if (L.vert) { *y = L.y1 + i * L.sx; *x = L.x1 + k * L.sy; }
    else        { *x = L.x1 + i * L.sx; *y = L.y1 + k * L.sy; }
}

}  // namespace raster
}  // namespace pn
