// P1 -- fused uint8 HWC BGR -> resize -> RGB -> x*(2/255)-1 -> f32 NCHW.
// Replaces posenet/utils.py:13-26 (_process_input) of the reference, i.e. cv2.resize(INTER_LINEAR) on
// uint8 + cvtColor + two rounded fp32 ops.  Integer/fixed-point work: bit-exact with OpenCV.
// HBM-bound: reads 3 B and writes 12 B per output pixel, x fastest.
#include "common.cuh"

namespace pn {

enum { MODE_COPY = 0, MODE_AREA2 = 1 };

// cv2: f = (float)((d + 0.5) * scale - 0.5) in double, s = floor(f), f -= s in fp32.  Explicit _rn
// intrinsics keep nvcc from contracting mul+add into an FMA (which rounds differently).
__device__ __forceinline__ void axis_coeff(int d, double scale, int &s, float &f) {
    f = (float)__dadd_rn(__dmul_rn(__dadd_rn((double)d, 0.5), scale), -0.5);
    float fl = floorf(f);
    s = (int)fl;
    f = __fsub_rn(f, fl);
}

__device__ __forceinline__ float normalise(int v) {
    // utils.py:23: input_img * (2.0 / 255.0) - 1.0 on float32 -> mul and sub each rounded to fp32
    return __fsub_rn(__fmul_rn((float)v, (float)(2.0 / 255.0)), 1.0f);
}

// OUT_U8: stop after the resize and keep uint8 BGR HWC (the tensor-core stem consumes that and normalises itself), so
// frames of any size can feed the uint8 fast path; otherwise the reference's normalised f32 RGB NCHW tensor.
// This kernel covers the same-size copy and the exact 2x decimation, one thread per output pixel; resize_linear_kernel the rest.
template <int MODE, bool OUT_U8>
__global__ void __launch_bounds__(256) preprocess_kernel(const uint8_t *__restrict__ src, void *__restrict__ dst_, int sh, int sw,
                                                          int dh, int dw) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y;
    const int img = blockIdx.z;
    if (x >= dw) return;
    const uint8_t *s = src + (size_t)img * sh * sw * 3;
    int bgr[3];
    if (MODE == MODE_COPY) {
        const uint8_t *p = s + ((size_t)y * sw + x) * 3;
        bgr[0] = p[0]; bgr[1] = p[1]; bgr[2] = p[2];
    } else {
        // exact 2x decimation takes cv2's INTER_AREA 2x2 box path
        const uint8_t *p0 = s + ((size_t)(2 * y) * sw + 2 * x) * 3;
        const uint8_t *p1 = p0 + (size_t)sw * 3;
#pragma unroll
        for (int c = 0; c < 3; ++c) bgr[c] = (p0[c] + p0[3 + c] + p1[c] + p1[3 + c] + 2) >> 2;
    }
    if (OUT_U8) {
        uint8_t *o8 = reinterpret_cast<uint8_t *>(dst_) + (((size_t)img * dh + y) * dw + x) * 3;
        o8[0] = (uint8_t)bgr[0]; o8[1] = (uint8_t)bgr[1]; o8[2] = (uint8_t)bgr[2];
        return;
    }
    const size_t plane = (size_t)dh * dw;
    float *o = reinterpret_cast<float *>(dst_) + (size_t)img * 3 * plane + (size_t)y * dw + x;
    o[0] = normalise(bgr[2]);          // utils.py:22 BGR -> RGB
    o[plane] = normalise(bgr[1]);
    o[2 * plane] = normalise(bgr[0]);
}

// cv2.resize INTER_LINEAR: a block covers 256 output columns x PRE_RB output rows; the row coefficients (float64 -> fixed point,
// the expensive part of a pixel) are computed once per block row into shared memory and the column coefficients once per thread,
// then reused down the rows.
constexpr int PRE_RB = 16;
template <bool OUT_U8>
__global__ void __launch_bounds__(256) resize_linear_kernel(const uint8_t *__restrict__ src, void *__restrict__ dst_, int sh, int sw,
                                                             int dh, int dw, double scale_x, double scale_y) {
    __shared__ int s_y0[PRE_RB], s_y1[PRE_RB], s_b0[PRE_RB], s_b1[PRE_RB];
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int ybase = blockIdx.y * PRE_RB;
    const int img = blockIdx.z;
    if (threadIdx.x < PRE_RB && ybase + threadIdx.x < dh) {
        int sy;
        float fy;
        axis_coeff(ybase + threadIdx.x, scale_y, sy, fy);              // rows: index clipped, weights kept
        s_y0[threadIdx.x] = min(max(sy, 0), sh - 1);
        s_y1[threadIdx.x] = min(max(sy + 1, 0), sh - 1);
        s_b1[threadIdx.x] = __float2int_rn(__fmul_rn(fy, 2048.f));
        s_b0[threadIdx.x] = __float2int_rn(__fmul_rn(__fsub_rn(1.f, fy), 2048.f));
    }
    __syncthreads();
    if (x >= dw) return;
    int sx;
    float fx;
    axis_coeff(x, scale_x, sx, fx);
    if (sx < 0) { sx = 0; fx = 0.f; }
    if (sx >= sw - 1) { sx = sw - 1; fx = 0.f; }
    const int x1 = min(sx + 1, sw - 1);
    const int a1 = __float2int_rn(__fmul_rn(fx, 2048.f));
    const int a0 = __float2int_rn(__fmul_rn(__fsub_rn(1.f, fx), 2048.f));
    const uint8_t *s = src + (size_t)img * sh * sw * 3;
    const int rows = min(PRE_RB, dh - ybase);
    const size_t plane = (size_t)dh * dw;
    // horizontal pass of a source row (cv2's int32 row sums); when the scale is near 1 the lower row of one output row is the
    // upper row of the next, so its sums are carried over instead of being recomputed from memory
    int carried_row = -1, hc[3] = {0, 0, 0};
    // (Three aligned 32-bit loads + funnel shifts for the six contiguous bytes of pixels sx, sx + 1 instead of six byte loads were
    // measured SLOWER: 138.7 vs 106.8 us for 32 frames of 1280 x 720 -- the byte loads of a warp coalesce in L1 and the extra
    // shifts / selects sit on the critical path; not kept.)
    auto hpass = [&](int row, int (&h)[3]) {
        const uint8_t *rp = s + (size_t)row * sw * 3;
#pragma unroll
        for (int c = 0; c < 3; ++c) h[c] = rp[sx * 3 + c] * a0 + rp[x1 * 3 + c] * a1;
    };
#pragma unroll 2
    for (int r = 0; r < rows; ++r) {
        const int y0 = s_y0[r], y1 = s_y1[r];
        const int b0 = s_b0[r], b1 = s_b1[r];
        int h0[3], h1[3];
        if (y0 == carried_row) { h0[0] = hc[0]; h0[1] = hc[1]; h0[2] = hc[2]; } else hpass(y0, h0);
        if (y1 == y0) { h1[0] = h0[0]; h1[1] = h0[1]; h1[2] = h0[2]; } else hpass(y1, h1);
        carried_row = y1; hc[0] = h1[0]; hc[1] = h1[1]; hc[2] = h1[2];
        int bgr[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const int v = (((b0 * (h0[c] >> 4)) >> 16) + ((b1 * (h1[c] >> 4)) >> 16) + 2) >> 2;
            bgr[c] = min(max(v, 0), 255);
        }
        const int y = ybase + r;
        if (OUT_U8) {
            uint8_t *o8 = reinterpret_cast<uint8_t *>(dst_) + (((size_t)img * dh + y) * dw + x) * 3;
            o8[0] = (uint8_t)bgr[0]; o8[1] = (uint8_t)bgr[1]; o8[2] = (uint8_t)bgr[2];
        } else {
            float *o = reinterpret_cast<float *>(dst_) + (size_t)img * 3 * plane + (size_t)y * dw + x;
            o[0] = normalise(bgr[2]);          // utils.py:22 BGR -> RGB
            o[plane] = normalise(bgr[1]);
            o[2 * plane] = normalise(bgr[0]);
        }
    }
}

template <bool OUT_U8>
static int launch_preprocess_t(const uint8_t *src, int n, int sh, int sw, int dh, int dw, void *dst, cudaStream_t st, const char *who) {
    PN_CHECK_ARG(src && dst && n > 0 && sh > 0 && sw > 0 && dh > 0 && dw > 0, "%s: bad argument", who);
    PN_CHECK_ARG(dh <= 65535 && n <= 65535, "%s: dst_h and n must be <= 65535", who);
    dim3 block(256), grid(ceil_div(dw, 256), dh, n);
    // cv2: inv_scale = dsize / ssize (double); scale = 1. / inv_scale
    const double scale_x = 1.0 / ((double)dw / (double)sw);
    const double scale_y = 1.0 / ((double)dh / (double)sh);
    if (dh == sh && dw == sw)
        preprocess_kernel<MODE_COPY, OUT_U8><<<grid, block, 0, st>>>(src, dst, sh, sw, dh, dw);
    else if (sh == 2 * dh && sw == 2 * dw)
        preprocess_kernel<MODE_AREA2, OUT_U8><<<grid, block, 0, st>>>(src, dst, sh, sw, dh, dw);
    else
        resize_linear_kernel<OUT_U8><<<dim3(ceil_div(dw, 256), ceil_div(dh, PRE_RB), n), block, 0, st>>>(src, dst, sh, sw, dh, dw, scale_x,
                                                                                                     scale_y);
    PN_CHECK_LAUNCH();
    return PN_OK;
}

int launch_preprocess(const uint8_t *src, int n, int sh, int sw, int dh, int dw, float *dst, cudaStream_t st) {
    return launch_preprocess_t<false>(src, n, sh, sw, dh, dw, dst, st, "pn_preprocess_u8");
}
int launch_resize_u8(const uint8_t *src, int n, int sh, int sw, int dh, int dw, uint8_t *dst, cudaStream_t st) {
    return launch_preprocess_t<true>(src, n, sh, sw, dh, dw, dst, st, "pn_resize_u8");
}

}  // namespace pn
