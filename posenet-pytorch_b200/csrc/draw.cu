// N4 (drawing half): posenet/utils.py draw_skel_and_kp / draw_skeleton for a batch of frames and pose records that are
// already on the device, bit-exact with cv2 (the arithmetic is draw_raster.cuh, shared with the host test).
//
// The frame is cut into 32x32 tiles and every tile has one owning warp.  Circles: the owner of a tile walks the keypoint
// list in order and draws every circle whose box touches the tile, one LineAA call after the other, the lanes of the warp
// taking the major-axis steps of a call that fall into the tile and writing only the tile's pixels.  So every pixel sees
// its blends in cv2's order (keypoint list order, then polygon segment order), and warps never share a pixel.  Segments
// come after a CTA barrier: they are one colour and overwrite, so any order works; a warp takes a segment, the lanes its
// pixels (LINE_8 in closed form), and a CTA writes only pixels of the tiles it owns, whose circles it has finished.
#include "common.cuh"
#include "draw_raster.cuh"

namespace pn {

namespace {

constexpr int TILE = 32;
constexpr int DRAW_WARPS = 8;
constexpr int MAX_POLY = 73;                   // 360 / 5 + 1 points (the smallest ellipse2Poly step)
constexpr int MAX_POSES = 512;                 // bounds the per-CTA circle table in shared memory

struct KpCircle {
    raster::Circle c;
    int selected;
};

struct DrawArgs {
    uint8_t *frames;
    long long frame_stride;
    const int *frame_hw;
    const double *pose_scores, *kp_scores, *kp_coords;
    int h, w, P, what;
    double min_pose, min_part;
};

struct Tile {
    int x0, y0, x1, y1;                        // [x0, x1) x [y0, y1), inside the frame
};

__device__ __forceinline__ bool box_hits(const Tile &t, long long bx0, long long by0, long long bx1, long long by1) {
    return bx1 >= t.x0 && bx0 < t.x1 && by1 >= t.y0 && by0 < t.y1;
}

// One LineAA call restricted to the pixels of tile t; the whole warp calls it with the same arguments.
__device__ void lineaa_tile(uint8_t *img, int fw, int fh, long long pitch, const Tile &t, int64_t x1, int64_t y1, int64_t x2,
                            int64_t y2, const uint8_t col[3]) {
    raster::LineAA L;
    if (!raster::lineaa_setup(fw, fh, x1, y1, x2, y2, L)) return;
    const int lane = threadIdx.x & 31;
    const int s = (L.x_major ? t.x0 : t.y0) + lane - L.start;
    if (s < 0 || s > L.ecount) return;
    int major, minor0, alpha[3];
    raster::lineaa_step(L, s, &major, &minor0, alpha);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const int x = L.x_major ? major : minor0 + k, y = L.x_major ? minor0 + k : major;
        if (x >= t.x0 && x < t.x1 && y >= t.y0 && y < t.y1) raster::blend_put(img + y * pitch + 3ll * x, col, alpha[k]);
    }
}

// EllipseEx: the polygon's points (deduplicated against their predecessor) joined by LineAA, inside tile t only.
__device__ void circle_tile(uint8_t *img, int fw, int fh, long long pitch, const Tile &t, const raster::Circle &c,
                            int64_t (*pts)[2], const uint8_t col[3]) {
    const int lane = threadIdx.x & 31;
    const raster::Poly p = raster::circle_poly(c);
    for (int k = lane; k < p.npts; k += 32) raster::poly_point(p, k, &pts[k][0], &pts[k][1]);
    __syncwarp();
    bool moved = false;
    for (int k = 1 + lane; k < p.npts; k += 32) moved |= pts[k][0] != pts[k - 1][0] || pts[k][1] != pts[k - 1][1];
    if (!__any_sync(0xffffffffu, moved)) {      // a single distinct point: cv2 draws the centre to itself
        lineaa_tile(img, fw, fh, pitch, t, p.cx, p.cy, p.cx, p.cy, col);
    } else {
        constexpr int M = 4;                   // px: covers the +1 end step, the +-1 footprint rows and the +1/2 bias
        for (int k = 1; k < p.npts; ++k) {
            const int64_t ax = pts[k - 1][0], ay = pts[k - 1][1], bx = pts[k][0], by = pts[k][1];
            if (ax == bx && ay == by) continue;
            const long long bx0 = ((ax < bx ? ax : bx) >> raster::XY_SHIFT) - M, bx1 = ((ax < bx ? bx : ax) >> raster::XY_SHIFT) + M;
            const long long by0 = ((ay < by ? ay : by) >> raster::XY_SHIFT) - M, by1 = ((ay < by ? by : ay) >> raster::XY_SHIFT) + M;
            if (!box_hits(t, bx0, by0, bx1, by1)) continue;
            lineaa_tile(img, fw, fh, pitch, t, ax, ay, bx, by, col);
            __syncwarp();                      // the next call may blend the same pixels (shared end points)
        }
    }
    __syncwarp();                              // pts is rewritten by the next circle
}

__global__ void __launch_bounds__(DRAW_WARPS * 32) draw_poses_kernel(DrawArgs a) {
    extern __shared__ __align__(16) unsigned char smem[];
    int64_t(*pts)[2] = reinterpret_cast<int64_t(*)[2]>(smem) + (threadIdx.x >> 5) * MAX_POLY;
    KpCircle *circ = reinterpret_cast<KpCircle *>(smem + sizeof(int64_t) * 2 * MAX_POLY * DRAW_WARPS);
    const uint8_t col[3] = {255, 255, 0};      // utils.py: color=(255, 255, 0), BGR
    const int img = blockIdx.y;
    const int fh = a.frame_hw ? a.frame_hw[2 * img] : a.h, fw = a.frame_hw ? a.frame_hw[2 * img + 1] : a.w;
    if (fh <= 0 || fw <= 0 || fh > a.h || fw > a.w) return;   // a row without a frame, or a size that would overrun it
    uint8_t *frame = a.frames + img * a.frame_stride;
    const long long pitch = 3ll * fw;
    const int tiles_x = (fw + TILE - 1) / TILE, tiles = tiles_x * ((fh + TILE - 1) / TILE);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool with_kp = (a.what & PN_DRAW_KEYPOINTS) != 0;
    const double *ps = a.pose_scores + (long long)img * a.P;
    const double *ks = a.kp_scores + (long long)img * a.P * PN_NUM_PARTS;
    const double *kc = a.kp_coords + (long long)img * a.P * PN_NUM_PARTS * 2;

    if (with_kp) {
        const int n = a.P * PN_NUM_PARTS;
        for (int q = threadIdx.x; q < n; q += blockDim.x) {
            KpCircle e;
            e.selected = raster::pose_selected(ps[q / PN_NUM_PARTS], a.min_pose, true) && ks[q] >= a.min_part;
            e.c = raster::keypoint_circle(kc[2 * q], kc[2 * q + 1], ks[q]);
            circ[q] = e;
        }
        __syncthreads();
        for (int ti = blockIdx.x + gridDim.x * warp; ti < tiles; ti += gridDim.x * DRAW_WARPS) {
            Tile t;
            t.x0 = (ti % tiles_x) * TILE; t.y0 = (ti / tiles_x) * TILE;
            t.x1 = min(t.x0 + TILE, fw); t.y1 = min(t.y0 + TILE, fh);
            for (int q0 = 0; q0 < n; q0 += 32) {
                bool hit = false;
                if (q0 + lane < n && circ[q0 + lane].selected) {
                    const raster::Poly p = raster::circle_poly(circ[q0 + lane].c);
                    constexpr int M = 6;       // px around cx +- r: point rounding plus the LineAA footprint
                    hit = box_hits(t, ((p.cx - p.r) >> raster::XY_SHIFT) - M, ((p.cy - p.r) >> raster::XY_SHIFT) - M,
                                   ((p.cx + p.r) >> raster::XY_SHIFT) + M, ((p.cy + p.r) >> raster::XY_SHIFT) + M);
                }
                unsigned mask = __ballot_sync(0xffffffffu, hit);
                while (mask) {
                    const int b = __ffs(mask) - 1;
                    mask &= mask - 1;
                    circle_tile(frame, fw, fh, pitch, t, circ[q0 + b].c, pts, col);
                }
            }
        }
        __syncthreads();                       // this CTA's tiles have all their circles: segments may overwrite them
    }
    if (a.what & PN_DRAW_SKELETON) {
        for (int sgi = warp; sgi < a.P * raster::NUM_LIMBS; sgi += DRAW_WARPS) {
            const int i = sgi / raster::NUM_LIMBS, e = sgi % raster::NUM_LIMBS;
            const int pa = raster::limb_part(e, 0), pb = raster::limb_part(e, 1);
            const double *kpa = ks + (long long)i * PN_NUM_PARTS, *kca = kc + (long long)i * PN_NUM_PARTS * 2;
            if (!(raster::pose_selected(ps[i], a.min_pose, with_kp) && kpa[pa] >= a.min_part && kpa[pb] >= a.min_part)) continue;
            raster::Line8 L;
            if (!raster::line8_setup(fw, fh, raster::trunc_i32(kca[2 * pa + 1]), raster::trunc_i32(kca[2 * pa]),
                                     raster::trunc_i32(kca[2 * pb + 1]), raster::trunc_i32(kca[2 * pb]), L))
                continue;
            for (int k = lane; k < L.count; k += 32) {
                int x, y;
                raster::line8_pixel(L, k, &x, &y);
                if ((unsigned)x >= (unsigned)fw || (unsigned)y >= (unsigned)fh) continue;
                if (((y / TILE) * tiles_x + x / TILE) % (int)gridDim.x != (int)blockIdx.x) continue;
                uint8_t *px = frame + y * pitch + 3ll * x;
                px[0] = col[0]; px[1] = col[1]; px[2] = col[2];
            }
        }
    }
}

}  // namespace

}  // namespace pn

using namespace pn;

extern "C" int pn_draw_poses(uint8_t *frames, int n_img, int h, int w, int64_t frame_stride, const int *frame_hw,
                             const double *pose_scores, const double *kp_scores, const double *kp_coords, int max_poses,
                             double min_pose_score, double min_part_score, int what, pn_stream_t stream) {
    PN_CHECK_ARG(frames && pose_scores && kp_scores && kp_coords, "pn_draw_poses: null pointer");
    PN_CHECK_ARG(n_img > 0 && n_img <= 65535, "pn_draw_poses: n_img %d out of 1..65535", n_img);
    PN_CHECK_ARG(h > 0 && w > 0 && h <= (1 << 24) && w <= (1 << 24), "pn_draw_poses: bad frame size %d x %d", h, w);
    PN_CHECK_ARG(frame_stride >= 3ll * h * w, "pn_draw_poses: frame_stride %lld < h*w*3", (long long)frame_stride);
    PN_CHECK_ARG(max_poses >= 0 && max_poses <= MAX_POSES, "pn_draw_poses: max_poses %d out of 0..%d", max_poses, MAX_POSES);
    PN_CHECK_ARG(what > 0 && (what & ~(PN_DRAW_KEYPOINTS | PN_DRAW_SKELETON)) == 0, "pn_draw_poses: bad what %d", what);
    if (max_poses == 0) return PN_OK;
    DrawArgs a;
    a.frames = frames; a.frame_stride = frame_stride; a.frame_hw = frame_hw;
    a.pose_scores = pose_scores; a.kp_scores = kp_scores; a.kp_coords = kp_coords;
    a.h = h; a.w = w; a.P = max_poses; a.what = what;
    a.min_pose = min_pose_score; a.min_part = min_part_score;
    const size_t smem = sizeof(int64_t) * 2 * MAX_POLY * DRAW_WARPS +
                        ((what & PN_DRAW_KEYPOINTS) ? sizeof(KpCircle) * max_poses * PN_NUM_PARTS : 0);
    static DeviceOnce once;
    const int dev = current_device();
    if (!once.get(dev)) {
        PN_CHECK_CUDA(cudaFuncSetAttribute(draw_poses_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)(sizeof(int64_t) * 2 * MAX_POLY * DRAW_WARPS + sizeof(KpCircle) * MAX_POSES * PN_NUM_PARTS)));
        once.set(dev, 1);
    }
    // CTAs per image: enough for two per SM over the batch, at most one per tile (the largest frame's tiles)
    const long long tiles = (long long)((h + TILE - 1) / TILE) * ((w + TILE - 1) / TILE);
    long long per_img = (2ll * num_sms() + n_img - 1) / n_img;
    if (per_img > tiles) per_img = tiles;
    if (per_img > 65535) per_img = 65535;
    draw_poses_kernel<<<dim3((unsigned)per_img, (unsigned)n_img), DRAW_WARPS * 32, smem, as_stream(stream)>>>(a);
    PN_CHECK_LAUNCH();
    return PN_OK;
}
