"""BGR -> YUV arithmetic (csrc/yuv_convert.cuh, the output half) against cv2.cvtColor, on the host.

The header is compiled into a small host library (a serial loop over the functions csrc/yuv.cu runs in parallel) and compared
with cv2 byte for byte.  cv2 runs two arithmetic families:
- 4:2:0 (I420 / YV12): a pixel's luma, and a 2x2 block's chroma from its top-left pixel alone.  One 8192 x 8192 frame whose
  2x2 blocks start with every one of the 2^24 BGR triples covers both; the other three pixels of a block are random, which
  shows they do not enter the chroma.
- 4:2:2 (YUY2 / UYVY / YVYU): a pixel's luma over all 2^24 triples, and a pair's chroma, which depends only on the pair's B, G
  and R sums.  Random pairs show that (a pair and another with the same sums give the same chroma); then every one of the
  511^3 sum triples is checked.
Also frame addressing at small and odd sizes, and the code / size checks of posenet.yuv and BatchPipeline(yuv_out=...), which
need no device.  The kernel's tiling and staging are covered by tests/test_gpu_yuv_out.py."""
import ctypes as C
import os
import subprocess

import cv2
import numpy as np
import pytest

import posenet
from posenet import _native as nat
from posenet import yuv

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "posenet-pytorch_b200", "csrc")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")

OUT_CODES = {                                                # every alias of the five layouts cv2 writes
    "I420": (nat.YUV_I420, ["COLOR_BGR2YUV_I420", "COLOR_BGR2YUV_IYUV"]),
    "YV12": (nat.YUV_YV12, ["COLOR_BGR2YUV_YV12"]),
    "YUY2": (nat.YUV_YUY2, ["COLOR_BGR2YUV_YUY2", "COLOR_BGR2YUV_YUYV", "COLOR_BGR2YUV_YUNV"]),
    "UYVY": (nat.YUV_UYVY, ["COLOR_BGR2YUV_UYVY", "COLOR_BGR2YUV_Y422", "COLOR_BGR2YUV_UYNV"]),
    "YVYU": (nat.YUV_YVYU, ["COLOR_BGR2YUV_YVYU"]),
}
OUT_LAYOUTS = list(OUT_CODES)

# frame sizes (h, w): 2x2, 2xN, Nx2, widths that are not multiples of 4, 16 or the kernel's 256-pixel tile, heights that are
# not multiples of its 8-row tile; 4:2:2 also takes odd heights
SIZES = [(2, 2), (2, 6), (2, 258), (6, 2), (34, 2), (4, 18), (10, 34), (18, 514), (46, 258), (14, 770), (720, 1280)]
SIZES_422 = [(1, 2), (1, 514), (3, 10), (9, 258), (17, 66), (33, 2)]

SHIM = r"""
#include "yuv_convert.cuh"
using namespace pn::yuv;
extern "C" void t_bgr_to_yuv(int layout, const uint8_t *bgr, int h, int w, uint8_t *out) {
    for (int y = 0; y < h; ++y) {
        const uint8_t *r0, *r1, *r2;
        frame_rows(layout, out, h, w, y, &r0, &r1, &r2);
        for (int x = 0; x < w; x += 2)
            put_pair(layout, bgr + (int64_t)y * w * 3, x, (y & 1) == 0, (uint8_t *)r0, (uint8_t *)r1, (uint8_t *)r2);
    }
}
"""


@pytest.fixture(scope="module")
def conv(tmp_path_factory):
    d = tmp_path_factory.mktemp("yuv_out")
    src, lib = d / "yuv_out_shim.cu", d / "libyuv_out_shim.so"
    src.write_text(SHIM)
    cmd = [NVCC, "-O2", "-std=c++17", "-shared", "-Xcompiler", "-fPIC", "-gencode", "arch=compute_100a,code=sm_100a",
           "-I", CSRC, str(src), "-o", str(lib)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    L = C.CDLL(str(lib))
    L.t_bgr_to_yuv.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    L.t_bgr_to_yuv.restype = None

    def run(layout, frame):
        frame = np.ascontiguousarray(frame)
        h, w = frame.shape[:2]
        out = np.empty(yuv.frame_shape(layout, h, w), np.uint8)
        L.t_bgr_to_yuv(layout, frame.ctypes.data, h, w, out.ctypes.data)
        return out
    return run


def code_of(name):
    return getattr(cv2, OUT_CODES[name][1][0])


def all_triples():
    """4096 x 4096 BGR frame holding every triple once."""
    k = np.arange(1 << 24, dtype=np.uint32)
    return np.stack([k & 255, (k >> 8) & 255, k >> 16], -1).astype(np.uint8).reshape(4096, 4096, 3)


def test_420_luma_and_chroma_over_every_triple(conv):
    """Block (i, j) of an 8192 x 8192 frame starts with triple 4096 i + j; its other three pixels are random."""
    rng = np.random.default_rng(1)
    frame = rng.integers(0, 256, (8192, 8192, 3), dtype=np.uint8)
    frame[0::2, 0::2] = all_triples()
    for name in ("I420", "YV12"):
        ref = cv2.cvtColor(frame, code_of(name))
        got = conv(OUT_CODES[name][0], frame)
        assert np.array_equal(got, ref), (name, int((got != ref).sum()))


def test_420_chroma_is_the_top_left_pixels():
    """The premise of the test above, against cv2 itself: changing the other three pixels of every block changes no U or V."""
    rng = np.random.default_rng(2)
    a = rng.integers(0, 256, (256, 512, 3), dtype=np.uint8)
    b = rng.integers(0, 256, a.shape, dtype=np.uint8)
    b[0::2, 0::2] = a[0::2, 0::2]
    ca, cb = (cv2.cvtColor(f, cv2.COLOR_BGR2YUV_I420) for f in (a, b))
    assert np.array_equal(ca[256:], cb[256:]) and not np.array_equal(ca[:256], cb[:256])


@pytest.mark.parametrize("name", ["YUY2", "UYVY", "YVYU"])
def test_422_luma_over_every_triple(conv, name):
    frame = all_triples()
    ref = cv2.cvtColor(frame, code_of(name))
    got = conv(OUT_CODES[name][0], frame)
    assert np.array_equal(got, ref), (name, int((got != ref).sum()))


def pair_frame(first, second):
    """[1, 2n, 3] frame of n pairs."""
    return np.stack([first, second], 1).reshape(1, -1, 3)


def test_422_chroma_depends_only_on_the_pair_sums():
    """4M random pairs against pairs with the same B, G and R sums, split differently, in cv2: same U and V everywhere."""
    rng = np.random.default_rng(3)
    n = 1 << 22
    p0 = rng.integers(0, 256, (n, 3), dtype=np.int64)
    p1 = rng.integers(0, 256, (n, 3), dtype=np.int64)
    s = p0 + p1
    q0 = rng.integers(np.maximum(s - 255, 0), np.minimum(s, 255) + 1)          # another split of the same sums
    q1 = s - q0
    assert (q0 != p0).any(1).mean() > 0.99
    a = cv2.cvtColor(pair_frame(p0, p1).astype(np.uint8).reshape(2048, -1, 3), cv2.COLOR_BGR2YUV_YUY2).reshape(n, 4)
    b = cv2.cvtColor(pair_frame(q0, q1).astype(np.uint8).reshape(2048, -1, 3), cv2.COLOR_BGR2YUV_YUY2).reshape(n, 4)
    assert np.array_equal(a[:, 1::2], b[:, 1::2])


def test_422_chroma_over_every_sum_triple(conv):
    """All 511^3 (sB, sG, sR) sums, each as the pair (min(s, 255), s - min(s, 255)), in chunks of 64 sR values: a frame of
    [64 * 511 rows (sR, sG), 511 pairs (sB)]."""
    s = np.arange(511)
    lo, hi = np.minimum(s, 255), s - np.minimum(s, 255)
    sb0, sb1 = np.broadcast_to(lo, (511, 511)), np.broadcast_to(hi, (511, 511))
    sg0, sg1 = np.broadcast_to(lo[:, None], (511, 511)), np.broadcast_to(hi[:, None], (511, 511))
    for r0 in range(0, 511, 64):
        rs = s[r0:r0 + 64]
        k = len(rs)
        frame = np.empty((k, 511, 511, 2, 3), np.uint8)
        frame[..., 0, 0], frame[..., 1, 0] = sb0, sb1
        frame[..., 0, 1], frame[..., 1, 1] = sg0, sg1
        frame[..., 0, 2] = np.minimum(rs, 255)[:, None, None]
        frame[..., 1, 2] = (rs - np.minimum(rs, 255))[:, None, None]
        frame = frame.reshape(k * 511, 1022, 3)
        for name in ("YUY2", "UYVY"):
            ref = cv2.cvtColor(frame, code_of(name))
            got = conv(OUT_CODES[name][0], frame)
            assert np.array_equal(got, ref), (name, r0, int((got != ref).sum()))


@pytest.mark.parametrize("name", OUT_LAYOUTS)
def test_saturation_corners(conv, name):
    """Every pair and 2x2 block of pixels from {0, 255}^3, and their mixes with 1, 16, 128, 235, 240 and 254."""
    vals = np.array([0, 1, 16, 128, 235, 240, 254, 255])
    corners = np.array(np.meshgrid(vals, vals, vals, indexing="ij")).reshape(3, -1).T
    a = np.repeat(corners, len(corners), 0)
    b = np.tile(corners, (len(corners), 1))
    frame = np.stack([np.stack([a, b], 1), np.stack([b, a], 1)], 0).reshape(2, -1, 3).astype(np.uint8)
    got = conv(OUT_CODES[name][0], frame)
    assert np.array_equal(got, cv2.cvtColor(frame, code_of(name))), name


@pytest.mark.parametrize("name", OUT_LAYOUTS)
def test_frame_addressing_matches_cv2(conv, name):
    layout = OUT_CODES[name][0]
    rng = np.random.default_rng(10 + layout)
    sizes = SIZES + [(2 * int(rng.integers(1, 40)), 2 * int(rng.integers(1, 300))) for _ in range(10)]
    if layout > nat.YUV_NV21:
        sizes += SIZES_422
    for h, w in sizes:
        frame = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        got = conv(layout, frame)
        assert np.array_equal(got, cv2.cvtColor(frame, code_of(name))), (name, h, w)


def test_layout_of_output_every_alias():
    for name, (layout, aliases) in OUT_CODES.items():
        for a in aliases:
            assert yuv.layout_of_output(getattr(cv2, a)) == layout, a
            assert yuv.layout_of_output(np.int64(getattr(cv2, a))) == layout, a


@pytest.mark.parametrize("code", [cv2.COLOR_BGR2YUV, cv2.COLOR_RGB2YUV_I420, cv2.COLOR_RGB2YUV_YUY2, cv2.COLOR_BGRA2YUV_I420,
                                  cv2.COLOR_BGRA2YUV_UYVY, cv2.COLOR_RGBA2YUV_YV12, cv2.COLOR_RGB2YUV_YVYU, cv2.COLOR_YUV2BGR_I420,
                                  cv2.COLOR_YUV2BGR_NV12, cv2.COLOR_BGR2GRAY, cv2.COLOR_BGR2YCrCb, -1, 1000, None, "I420", 128.0,
                                  True])
def test_other_codes_raise(code):
    with pytest.raises(ValueError):
        yuv.layout_of_output(code)
    with pytest.raises(ValueError):
        posenet.bgr_to_yuv_batch(np.zeros((1, 4, 4, 3), np.uint8), code)


def test_sizes_and_shapes_cv2_rejects_raise():
    i420, yuy2 = cv2.COLOR_BGR2YUV_I420, cv2.COLOR_BGR2YUV_YUY2
    for shape, code in [((1, 4, 5, 3), i420), ((1, 5, 4, 3), i420), ((1, 3, 2, 3), cv2.COLOR_BGR2YUV_YV12), ((1, 4, 5, 3), yuy2),
                        ((1, 1, 3, 3), cv2.COLOR_BGR2YUV_UYVY), ((1, 0, 4, 3), yuy2), ((1, 4, 0, 3), i420)]:
        frame = np.zeros(shape, np.uint8)
        with pytest.raises(cv2.error):
            cv2.cvtColor(frame[0], code)
        with pytest.raises(ValueError):
            posenet.bgr_to_yuv_batch(frame, code)
    for shape in [(1, 4, 4), (1, 4, 4, 4), (4, 4, 3), (1, 4, 4, 1)]:
        with pytest.raises(ValueError):
            posenet.bgr_to_yuv_batch(np.zeros(shape, np.uint8), i420)
    with pytest.raises(ValueError):
        posenet.bgr_to_yuv_batch(np.zeros((1, 4, 4, 3), np.int16), i420)
    assert cv2.cvtColor(np.zeros((5, 4, 3), np.uint8), yuy2).shape == yuv.frame_shape(nat.YUV_YUY2, 5, 4) == (5, 4, 2)
    assert cv2.cvtColor(np.zeros((4, 6, 3), np.uint8), i420).shape == yuv.frame_shape(nat.YUV_I420, 4, 6) == (6, 6)


def test_pipeline_rejects_bad_yuv_out():
    """Checked before anything touches the model or the device."""
    i420, yuy2, ov = cv2.COLOR_BGR2YUV_I420, cv2.COLOR_BGR2YUV_YUY2, (0.1, 0.1)
    bad = [dict(yuv_out=i420),                                               # no overlay
           dict(yuv_out=i420, overlay=ov, encode=[]),
           dict(yuv_out=yuy2, overlay=ov, encode=[], encode_ext=".png"),
           dict(yuv_out=i420, overlay=ov, mixed=True),
           dict(yuv_out=yuy2, overlay=ov, mixed=True, source_coords=True),
           dict(yuv_out=cv2.COLOR_YUV2BGR_I420, overlay=ov),
           dict(yuv_out=cv2.COLOR_RGB2YUV_I420, overlay=ov),
           dict(yuv_out=cv2.COLOR_BGR2YUV, overlay=ov)]
    for kw in bad:
        with pytest.raises(ValueError):
            posenet.BatchPipeline(None, 2, 720, 1280, **kw)
    for code, h, w in ((i420, 721, 1280), (i420, 720, 1281), (cv2.COLOR_BGR2YUV_YV12, 3, 4), (yuy2, 720, 1281),
                       (cv2.COLOR_BGR2YUV_YVYU, 5, 7)):
        with pytest.raises(ValueError):
            posenet.BatchPipeline(None, 2, h, w, overlay=ov, yuv_out=code)
