// N7: video frames in YUV 4:2:0 / 4:2:2 converted to BGR on the device, bit-exact with cv2.cvtColor(COLOR_YUV2BGR_<layout>)
// (the arithmetic is yuv_convert.cuh, shared with the host test).
//
// The kernel only moves bytes: 1.5 or 2 B/px in, 3 B/px out.  A CTA owns a tile of ROW_PAIRS row pairs x TILE_W pixels of one
// frame.  It copies the tile's source rows into shared memory with aligned 16-byte loads (each row lands at its global address
// mod 16, so the bytes of an unaligned row start or end are the only byte loads), converts there -- one thread per 2x2 group of
// 4:2:0, per horizontal pair of each row of 4:2:2 -- and writes the BGR rows back the same way, as full 16-byte stores.  3-byte
// pixels stored one by one would leave most store sectors partly used (DESIGN.md section 3, the stem note).
#include "common.cuh"
#include "yuv_convert.cuh"

namespace pn {

namespace {

constexpr int YUV_THREADS = 128;
constexpr int TILE_W = 2 * YUV_THREADS;         // pixels: a pixel pair per thread
constexpr int ROW_PAIRS = 4;                    // row pairs per tile: 24-32 bytes of loads in flight per thread
constexpr int ROWS = 2 * ROW_PAIRS;
constexpr int R0_SLOT = 2 * TILE_W + 32;        // shared bytes of one staged row: 15 bytes of alignment lead + the row
constexpr int C_SLOT = TILE_W + 32;
constexpr int OUT_SLOT = 3 * TILE_W + 32;
constexpr int IN_SEGS = ROWS + 2 * ROW_PAIRS;   // r0 of every row, r1 and r2 of every row pair
constexpr int WARPS = YUV_THREADS / 32;

struct YuvArgs {
    const uint8_t *src;
    uint8_t *dst;
    long long src_stride, dst_stride;
    int h, w;
};

// A row segment [g, g + n) staged at slot + lead (lead = g mod 16), so the 16-byte blocks of global and shared memory line up.
// A warp copies a segment, a lane a block; a block not wholly inside the segment is copied byte by byte, so nothing outside
// it is touched.
struct Seg {
    uint8_t *g;
    uint8_t *slot;
    int n, lead;
};

__device__ __forceinline__ int seg_blocks(const Seg &s) { return s.n > 0 ? (s.lead + s.n + 15) >> 4 : 0; }

template <int L>
__global__ void __launch_bounds__(YUV_THREADS, 12) yuv_to_bgr_kernel(YuvArgs a) {
    __shared__ __align__(16) uint8_t s_r0[ROWS][R0_SLOT];
    __shared__ __align__(16) uint8_t s_c[2][ROW_PAIRS][C_SLOT];
    __shared__ __align__(16) uint8_t s_out[ROWS][OUT_SLOT];
    __shared__ int s_lead[IN_SEGS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int x0 = blockIdx.x * TILE_W, y0 = blockIdx.y * ROWS;
    const int npix = min(TILE_W, a.w - x0);
    const uint8_t *frame = a.src + blockIdx.z * a.src_stride;

    // segment k: r0 of row k (k < ROWS), else r1 / r2 of row pair (k - ROWS) % ROW_PAIRS
    auto in_seg = [&](int k) {
        Seg s;
        const int which = k < ROWS ? 0 : 1 + (k - ROWS) / ROW_PAIRS;
        const int row = k < ROWS ? k : 2 * ((k - ROWS) % ROW_PAIRS);
        s.n = 0;
        s.slot = k < ROWS ? s_r0[k] : s_c[which - 1][(k - ROWS) % ROW_PAIRS];
        if (y0 + row < a.h) {
            const uint8_t *r[3];
            yuv::frame_rows(L, frame, a.h, a.w, y0 + row, &r[0], &r[1], &r[2]);
            s.g = const_cast<uint8_t *>(r[which]) + yuv::row_bytes(L, which, x0);
            s.n = yuv::row_bytes(L, which, npix);
        }
        s.lead = s.n > 0 ? (int)(reinterpret_cast<uintptr_t>(s.g) & 15) : 0;
        return s;
    };

    // ---- stage the source rows: every lane issues all its 16-byte loads before it stores any
    constexpr int IN_PER_WARP = IN_SEGS / WARPS;
    Seg segs[IN_PER_WARP];
    uint4 v[IN_PER_WARP][2];
#pragma unroll
    for (int j = 0; j < IN_PER_WARP; ++j) {
        const Seg s = segs[j] = in_seg(warp + WARPS * j);
        if (lane == 0) s_lead[warp + WARPS * j] = s.lead;
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const int off = 16 * (lane + 32 * q) - s.lead;
            if (off >= 0 && off + 16 <= s.n) v[j][q] = __ldg(reinterpret_cast<const uint4 *>(s.g + off));
        }
    }
#pragma unroll
    for (int j = 0; j < IN_PER_WARP; ++j) {
        const Seg &s = segs[j];
        const int nb = seg_blocks(s);
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const int blk = lane + 32 * q, off = 16 * blk - s.lead;
            if (blk >= nb) continue;
            if (off >= 0 && off + 16 <= s.n) {
                *reinterpret_cast<uint4 *>(s.slot + 16 * blk) = v[j][q];
            } else {
                for (int b = 0; b < 16; ++b)
                    if (off + b >= 0 && off + b < s.n) s.slot[16 * blk + b] = s.g[off + b];
            }
        }
    }
    __syncthreads();

    // ---- convert: thread t owns pixels 2t, 2t + 1 of every row of the tile
    const int xl = 2 * threadIdx.x;
    if (xl < npix) {
#pragma unroll
        for (int p = 0; p < ROW_PAIRS; ++p) {
            if (y0 + 2 * p >= a.h) break;
            const uint8_t *r1 = s_c[0][p] + s_lead[ROWS + p], *r2 = s_c[1][p] + s_lead[ROWS + ROW_PAIRS + p];
            yuv::Chroma c;
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int row = 2 * p + j;
                if (y0 + row >= a.h) break;             // the odd last row of a 4:2:2 frame
                const uint8_t *r0 = s_r0[row] + s_lead[row];
                int Y0, Y1, U, V;
                yuv::sample(L, r0, r1, r2, xl, &Y0, &U, &V);
                yuv::sample(L, r0, r1, r2, xl + 1, &Y1, &U, &V);
                if (j == 0 || !yuv::is_420(L)) c = yuv::chroma(U, V);
                uint8_t *o = a.dst + blockIdx.z * a.dst_stride + ((long long)(y0 + row) * a.w + x0) * 3;
                uint8_t *so = s_out[row] + (reinterpret_cast<uintptr_t>(o) & 15) + 3 * xl;
                yuv::pixel(Y0, c, so);
                yuv::pixel(Y1, c, so + 3);
            }
        }
    }
    __syncthreads();

    // ---- write the BGR rows back, two per warp
#pragma unroll
    for (int j = 0; j < ROWS / WARPS; ++j) {
        const int row = warp + WARPS * j;
        if (y0 + row >= a.h) continue;
        Seg s;
        s.g = a.dst + blockIdx.z * a.dst_stride + ((long long)(y0 + row) * a.w + x0) * 3;
        s.slot = s_out[row];
        s.n = 3 * npix;
        s.lead = (int)(reinterpret_cast<uintptr_t>(s.g) & 15);
        const int nb = seg_blocks(s);
        for (int blk = lane; blk < nb; blk += 32) {
            const int off = 16 * blk - s.lead;
            if (off >= 0 && off + 16 <= s.n) {
                *reinterpret_cast<uint4 *>(s.g + off) = *reinterpret_cast<const uint4 *>(s.slot + 16 * blk);
            } else {
                for (int b = 0; b < 16; ++b)
                    if (off + b >= 0 && off + b < s.n) s.g[off + b] = s.slot[16 * blk + b];
            }
        }
    }
}

}  // namespace

}  // namespace pn

using namespace pn;

extern "C" int pn_yuv_to_bgr(const uint8_t *src, int n_img, int h, int w, int64_t src_stride, int layout, uint8_t *dst,
                             int64_t dst_stride, pn_stream_t stream) {
    PN_CHECK_ARG(src && dst, "pn_yuv_to_bgr: null pointer");
    PN_CHECK_ARG(n_img > 0 && n_img <= 65535, "pn_yuv_to_bgr: n_img %d out of 1..65535", n_img);
    PN_CHECK_ARG(layout >= PN_YUV_I420 && layout <= PN_YUV_YVYU, "pn_yuv_to_bgr: unknown layout %d", layout);
    PN_CHECK_ARG(h > 0 && w > 0 && w % 2 == 0 && (h % 2 == 0 || !yuv::is_420(layout)) && h <= (1 << 18) && w <= (1 << 18),
                 "pn_yuv_to_bgr: frame size %d x %d: the width must be even, and the height too for 4:2:0", h, w);
    PN_CHECK_ARG(src_stride >= yuv::frame_bytes(layout, h, w), "pn_yuv_to_bgr: src_stride %lld < the frame's %lld bytes",
                 (long long)src_stride, (long long)yuv::frame_bytes(layout, h, w));
    PN_CHECK_ARG(dst_stride >= 3ll * h * w, "pn_yuv_to_bgr: dst_stride %lld < h*w*3", (long long)dst_stride);
    YuvArgs a;
    a.src = src; a.dst = dst; a.src_stride = src_stride; a.dst_stride = dst_stride; a.h = h; a.w = w;
    const dim3 grid(ceil_div(w, TILE_W), ceil_div(h, ROWS), n_img);
    const cudaStream_t st = as_stream(stream);
    switch (layout) {
    case PN_YUV_I420: yuv_to_bgr_kernel<PN_YUV_I420><<<grid, YUV_THREADS, 0, st>>>(a); break;
    case PN_YUV_YV12: yuv_to_bgr_kernel<PN_YUV_YV12><<<grid, YUV_THREADS, 0, st>>>(a); break;
    case PN_YUV_NV12: yuv_to_bgr_kernel<PN_YUV_NV12><<<grid, YUV_THREADS, 0, st>>>(a); break;
    case PN_YUV_NV21: yuv_to_bgr_kernel<PN_YUV_NV21><<<grid, YUV_THREADS, 0, st>>>(a); break;
    case PN_YUV_YUY2: yuv_to_bgr_kernel<PN_YUV_YUY2><<<grid, YUV_THREADS, 0, st>>>(a); break;
    case PN_YUV_UYVY: yuv_to_bgr_kernel<PN_YUV_UYVY><<<grid, YUV_THREADS, 0, st>>>(a); break;
    default:          yuv_to_bgr_kernel<PN_YUV_YVYU><<<grid, YUV_THREADS, 0, st>>>(a); break;
    }
    PN_CHECK_LAUNCH();
    return PN_OK;
}
