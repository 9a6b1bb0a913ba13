"""The overlay rasteriser (csrc/draw_raster.cuh) against cv2, on the host.

The header is compiled into a small host library (serial loops over the same functions csrc/draw.cu runs in parallel) and
compared with cv2.drawKeypoints / cv2.polylines / cv2.line and with posenet.draw_skel_and_kp / draw_skeleton, byte for
byte.  The parallel decomposition of the kernel (tiles, lanes) is covered by tests/test_gpu_draw.py."""
import ctypes as C
import os
import subprocess

import cv2
import numpy as np
import pytest

import posenet

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "posenet-pytorch_b200", "csrc")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
COLOR = (255, 255, 0)

SHIM = r"""
#include "draw_raster.cuh"
using namespace pn::raster;
static const uint8_t kCol[3] = {255, 255, 0};

static void lineaa(uint8_t *img, int h, int w, int64_t x1, int64_t y1, int64_t x2, int64_t y2) {
    LineAA L;
    if (!lineaa_setup(w, h, x1, y1, x2, y2, L)) return;
    for (int s = 0; s <= L.ecount; ++s) {
        int major, minor0, alpha[3];
        lineaa_step(L, s, &major, &minor0, alpha);
        if ((unsigned)major >= (unsigned)(L.x_major ? w : h)) continue;
        for (int k = 0; k < 3; ++k) {
            const int x = L.x_major ? major : minor0 + k, y = L.x_major ? minor0 + k : major;
            if ((unsigned)x < (unsigned)w && (unsigned)y < (unsigned)h) blend_put(img + ((int64_t)y * w + x) * 3, kCol, alpha[k]);
        }
    }
}

static void circle(uint8_t *img, int h, int w, const Circle &c) {
    const Poly p = circle_poly(c);
    int64_t pts[80][2];
    for (int k = 0; k < p.npts; ++k) poly_point(p, k, &pts[k][0], &pts[k][1]);
    int drawn = 0;
    for (int k = 1; k < p.npts; ++k) {
        if (pts[k][0] == pts[k - 1][0] && pts[k][1] == pts[k - 1][1]) continue;
        lineaa(img, h, w, pts[k - 1][0], pts[k - 1][1], pts[k][0], pts[k][1]);
        ++drawn;
    }
    if (!drawn) lineaa(img, h, w, p.cx, p.cy, p.cx, p.cy);
}

static void line8(uint8_t *img, int h, int w, int x1, int y1, int x2, int y2) {
    Line8 L;
    if (!line8_setup(w, h, x1, y1, x2, y2, L)) return;
    for (int i = 0; i < L.count; ++i) {
        int x, y;
        line8_pixel(L, i, &x, &y);
        if ((unsigned)x < (unsigned)w && (unsigned)y < (unsigned)h)
            for (int c = 0; c < 3; ++c) img[((int64_t)y * w + x) * 3 + c] = kCol[c];
    }
}

extern "C" {
void t_lineaa(uint8_t *img, int h, int w, long long x1, long long y1, long long x2, long long y2) { lineaa(img, h, w, x1, y1, x2, y2); }
void t_line8(uint8_t *img, int h, int w, int x1, int y1, int x2, int y2) { line8(img, h, w, x1, y1, x2, y2); }
// draw_skel_and_kp (what = 3) / draw_skeleton (what = 2) / the circles alone (what = 1) of one image, serially
void t_draw_poses(uint8_t *img, int h, int w, const double *ps, const double *ks, const double *kc, int P, double mp, double mk,
                  int what) {
    const bool with_kp = what & 1;
    if (with_kp)
        for (int q = 0; q < P * 17; ++q)
            if (pose_selected(ps[q / 17], mp, true) && ks[q] >= mk) circle(img, h, w, keypoint_circle(kc[2 * q], kc[2 * q + 1], ks[q]));
    if (what & 2)
        for (int i = 0; i < P; ++i)
            for (int e = 0; e < NUM_LIMBS; ++e) {
                const int a = i * 17 + limb_part(e, 0), b = i * 17 + limb_part(e, 1);
                if (pose_selected(ps[i], mp, with_kp) && ks[a] >= mk && ks[b] >= mk)
                    line8(img, h, w, trunc_i32(kc[2 * a + 1]), trunc_i32(kc[2 * a]), trunc_i32(kc[2 * b + 1]), trunc_i32(kc[2 * b]));
            }
}
}
"""


@pytest.fixture(scope="module")
def raster(tmp_path_factory):
    d = tmp_path_factory.mktemp("raster")
    src, lib = d / "raster_shim.cu", d / "libraster_shim.so"
    src.write_text(SHIM)
    cmd = [NVCC, "-O2", "-std=c++17", "-shared", "-Xcompiler", "-fPIC", "-gencode", "arch=compute_100a,code=sm_100a",
           "-I", CSRC, str(src), "-o", str(lib)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    L = C.CDLL(str(lib))
    u8, i, ll, d_ = C.c_void_p, C.c_int, C.c_longlong, C.c_double
    L.t_lineaa.argtypes = [u8, i, i, ll, ll, ll, ll]
    L.t_line8.argtypes = [u8, i, i, i, i, i, i]
    L.t_draw_poses.argtypes = [u8, i, i, u8, u8, u8, i, d_, d_, i]
    return L


def _ptr(a):
    return C.c_void_p(a.ctypes.data)


def draw_poses(L, img, ps, ks, kc, mp, mk, what):
    out = np.ascontiguousarray(img.copy())
    ps, ks, kc = (np.ascontiguousarray(a, dtype=np.float64) for a in (ps, ks, kc))
    L.t_draw_poses(_ptr(out), out.shape[0], out.shape[1], _ptr(ps), _ptr(ks), _ptr(kc), ps.shape[0], mp, mk, what)
    return out


def test_keypoint_circles_match_drawkeypoints(raster):
    """Random rich keypoints: off-frame, radius 0, overlapping, sizes up to 60 (all four ellipse2Poly steps)."""
    rng = np.random.default_rng(11)
    deltas = set()
    for t in range(300):
        h, w = int(rng.integers(5, 41)), int(rng.integers(5, 41))
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        n = int(rng.integers(1, 40))
        pts = np.stack([rng.uniform(-15, h + 15, n), rng.uniform(-15, w + 15, n)], -1)      # (y, x)
        if t % 3 == 0:
            pts[n // 2:] = pts[0] + rng.uniform(-2, 2, (n - n // 2, 2))                      # a cluster of overlapping circles
        pts[: n // 3] = np.round(pts[: n // 3] * 32) / 32                                   # exact 1/32 px boundaries
        scores = rng.uniform(0, 6, n)
        scores[rng.uniform(size=n) < 0.15] = 0.0                                              # radius 0
        scores[rng.uniform(size=n) < 0.15] = rng.uniform(0, 0.06)                             # sub-pixel radii
        for s in scores:
            r = abs(int(np.rint(np.float32(np.float32(10.0 * s) / 2) * 16))) << 12
            d = (r + 32768) >> 16
            deltas.add(90 if d < 3 else 30 if d < 10 else 18 if d < 15 else 5)
        kps = [cv2.KeyPoint(float(x), float(y), 10. * float(s)) for (y, x), s in zip(pts, scores)]
        ref = cv2.drawKeypoints(img, kps, outImage=np.array([]), color=COLOR, flags=cv2.DRAW_MATCHES_FLAGS_DRAW_RICH_KEYPOINTS)
        P = (n + 16) // 17                                                                   # packed as poses of 17 parts
        ks = np.full(P * 17, -1.0)
        kc = np.zeros((P * 17, 2))
        ks[:n], kc[:n] = scores, pts
        got = draw_poses(raster, img, np.ones(P), ks.reshape(P, 17), kc.reshape(P, 17, 2), 0.0, 0.0, 1)
        assert np.array_equal(got, ref), t
    assert deltas == {90, 30, 18, 5}


def test_line8_polylines_match_cv2(raster):
    rng = np.random.default_rng(12)
    for t in range(2000):
        h, w = int(rng.integers(1, 50)), int(rng.integers(1, 50))
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        p = np.stack([rng.integers(-60, w + 60, 2), rng.integers(-60, h + 60, 2)], -1).astype(np.int32)
        if t % 5 == 0:
            p *= rng.integers(1, 1 << 14)                                                    # far off the frame
        ref = cv2.polylines(img.copy(), [p], isClosed=False, color=COLOR)
        got = img.copy()
        raster.t_line8(_ptr(got), h, w, int(p[0, 0]), int(p[0, 1]), int(p[1, 0]), int(p[1, 1]))
        assert np.array_equal(got, ref), (t, p.tolist(), h, w)


def test_lineaa_matches_cv2(raster):
    """LineAA in 16.16 fixed point (cv2.line LINE_AA with shift 16), clipped and unclipped."""
    rng = np.random.default_rng(13)
    for t in range(2000):
        h, w = int(rng.integers(1, 40)), int(rng.integers(1, 40))
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        p = np.stack([rng.integers(-20 << 16, (w + 20) << 16, 2), rng.integers(-20 << 16, (h + 20) << 16, 2)], -1)
        if t % 7 == 0:
            p[1] = p[0] + rng.integers(-3 << 16, 3 << 16, 2)                                 # short, like a circle's sides
        ref = cv2.line(img.copy(), tuple(int(v) for v in p[0]), tuple(int(v) for v in p[1]), COLOR, 1, cv2.LINE_AA, 16)
        got = img.copy()
        raster.t_lineaa(_ptr(got), h, w, int(p[0, 0]), int(p[0, 1]), int(p[1, 0]), int(p[1, 1]))
        assert np.array_equal(got, ref), (t, p.tolist(), h, w)


@pytest.mark.parametrize("shape", [(513, 513), (720, 1280), (257, 257), (33, 47)])
def test_composites_match_draw_skel_and_kp(raster, shape):
    rng = np.random.default_rng(shape[0] * 7 + shape[1])
    h, w = shape
    for t in range(6):
        P = (10, 50)[t % 2]
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        ps = np.where(rng.uniform(size=P) < 0.8, np.sort(rng.uniform(0, 1, P))[::-1], 0.)
        ks = rng.uniform(0, 1, (P, 17))
        ks[rng.uniform(size=(P, 17)) < 0.1] = 0.25                                           # scores exactly at a threshold
        kc = np.stack([rng.uniform(-20, h + 20, (P, 17)), rng.uniform(-20, w + 20, (P, 17))], -1)
        kc[:, :5] = np.round(kc[:, :5] * 32) / 32
        mp, mk = [(0.25, 0.25), (0., 0.), (0.5, 0.5)][t % 3]
        ref = posenet.draw_skel_and_kp(img.copy(), ps, ks, kc, mp, mk)
        assert np.array_equal(draw_poses(raster, img, ps, ks, kc, mp, mk, 3), ref), (shape, t)
        ref = posenet.draw_skeleton(img.copy(), ps, ks, kc, mp, mk)
        assert np.array_equal(draw_poses(raster, img, ps, ks, kc, mp, mk, 2), ref), (shape, t)


def test_large_coordinates_match_cv2(raster):
    """Keypoints up to 2^26 px away from a small frame: the fixed-point ranges hold and nothing is drawn wrongly."""
    rng = np.random.default_rng(14)
    for t in range(40):
        img = rng.integers(0, 256, (40, 50, 3), dtype=np.uint8)
        ks = rng.uniform(0.3, 1, (3, 17))
        kc = rng.uniform(-(1 << 26), 1 << 26, (3, 17, 2)) * rng.choice([1.0, 1e-5], (3, 17, 2))
        ref = posenet.draw_skel_and_kp(img.copy(), np.ones(3), ks, kc, 0.1, 0.1)
        assert np.array_equal(draw_poses(raster, img, np.ones(3), ks, kc, 0.1, 0.1, 3), ref), t
