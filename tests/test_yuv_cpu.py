"""YUV -> BGR arithmetic (csrc/yuv_convert.cuh) against cv2.cvtColor, on the host.

The header is compiled into a small host library (a serial loop over the functions csrc/yuv.cu runs in parallel) and compared
with cv2 byte for byte: exhaustively over every (Y, U, V) triple for each of the seven layouts, and over random frame sizes.
Also the code / shape checks of posenet.yuv and BatchPipeline(yuv=...), which need no device.  The kernel's tiling and staging
are covered by tests/test_gpu_yuv.py."""
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

CODES = {                                                    # every alias of the seven layouts
    "I420": (nat.YUV_I420, ["COLOR_YUV2BGR_I420", "COLOR_YUV2BGR_IYUV"]),
    "YV12": (nat.YUV_YV12, ["COLOR_YUV2BGR_YV12"]),
    "NV12": (nat.YUV_NV12, ["COLOR_YUV2BGR_NV12"]),
    "NV21": (nat.YUV_NV21, ["COLOR_YUV2BGR_NV21"]),
    "YUY2": (nat.YUV_YUY2, ["COLOR_YUV2BGR_YUY2", "COLOR_YUV2BGR_YUYV", "COLOR_YUV2BGR_YUNV"]),
    "UYVY": (nat.YUV_UYVY, ["COLOR_YUV2BGR_UYVY", "COLOR_YUV2BGR_Y422", "COLOR_YUV2BGR_UYNV"]),
    "YVYU": (nat.YUV_YVYU, ["COLOR_YUV2BGR_YVYU"]),
}
LAYOUTS = list(CODES)

SHIM = r"""
#include "yuv_convert.cuh"
using namespace pn::yuv;
extern "C" void t_yuv_to_bgr(int layout, const uint8_t *f, int h, int w, uint8_t *out) {
    for (int y = 0; y < h; ++y) {
        const uint8_t *r0, *r1, *r2;
        frame_rows(layout, f, h, w, y, &r0, &r1, &r2);
        for (int x = 0; x < w; ++x) {
            int Y, U, V;
            sample(layout, r0, r1, r2, x, &Y, &U, &V);
            pixel(Y, chroma(U, V), out + ((int64_t)y * w + x) * 3);
        }
    }
}
"""


@pytest.fixture(scope="module")
def conv(tmp_path_factory):
    d = tmp_path_factory.mktemp("yuv")
    src, lib = d / "yuv_shim.cu", d / "libyuv_shim.so"
    src.write_text(SHIM)
    cmd = [NVCC, "-O2", "-std=c++17", "-shared", "-Xcompiler", "-fPIC", "-gencode", "arch=compute_100a,code=sm_100a",
           "-I", CSRC, str(src), "-o", str(lib)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    L = C.CDLL(str(lib))
    L.t_yuv_to_bgr.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    L.t_yuv_to_bgr.restype = None

    def run(layout, frame, h, w):
        frame = np.ascontiguousarray(frame)
        out = np.empty((h, w, 3), np.uint8)
        L.t_yuv_to_bgr(layout, frame.ctypes.data, h, w, out.ctypes.data)
        return out
    return run


def pack(name, Y, U, V):
    """cv2's input frame of layout `name` from planes Y [h, w] and U, V [h/2, w/2] (4:2:0) or [h, w/2] (4:2:2)."""
    h, w = Y.shape
    if name in ("I420", "YV12"):
        a, b = (U, V) if name == "I420" else (V, U)
        return np.concatenate([Y.ravel(), a.ravel(), b.ravel()]).reshape(h * 3 // 2, w)
    if name in ("NV12", "NV21"):
        a, b = (U, V) if name == "NV12" else (V, U)
        return np.concatenate([Y, np.stack([a, b], -1).reshape(h // 2, w)]).reshape(h * 3 // 2, w)
    y0, y1 = Y[:, 0::2], Y[:, 1::2]
    quad = {"YUY2": (y0, U, y1, V), "UYVY": (U, y0, V, y1), "YVYU": (y0, V, y1, U)}[name]
    return np.stack(quad, -1).reshape(h, w, 2)


def code_of(name):
    return getattr(cv2, CODES[name][1][0])


@pytest.mark.parametrize("name", LAYOUTS)
def test_every_yuv_triple_matches_cv2(conv, name):
    """One frame holds all 2^24 (Y, U, V) triples.  4:2:0 (4096 x 4096): 2x2 block k has (U, V) = k & 0xFFFF and luma
    4 * (k >> 16) + 0..3.  4:2:2 (2048 x 8192): pair k has (U, V) = k & 0xFFFF and luma 2 * (k >> 16) + 0..1."""
    layout = CODES[name][0]
    if layout <= nat.YUV_NV21:
        h = w = 4096
        k = np.arange(h // 2 * (w // 2), dtype=np.int64).reshape(h // 2, w // 2)
        U, V = (k & 0xFF).astype(np.uint8), ((k >> 8) & 0xFF).astype(np.uint8)
        base = 4 * (k >> 16)
        Y = np.empty((h, w), np.uint8)
        for dy in range(2):
            for dx in range(2):
                Y[dy::2, dx::2] = base + 2 * dy + dx
    else:
        h, w = 2048, 8192
        k = np.arange(h * (w // 2), dtype=np.int64).reshape(h, w // 2)
        U, V = (k & 0xFF).astype(np.uint8), ((k >> 8) & 0xFF).astype(np.uint8)
        Y = np.repeat(2 * (k >> 16), 2, axis=1) + np.tile([0, 1], w // 2)
        Y = Y.astype(np.uint8)
    triples = (Y.astype(np.int64) << 16) | (np.repeat(np.repeat(U, 2, 1), 2 if layout <= nat.YUV_NV21 else 1, 0).astype(np.int64)
                                            << 8) | np.repeat(np.repeat(V, 2, 1), 2 if layout <= nat.YUV_NV21 else 1, 0)
    assert np.unique(triples).size == 1 << 24
    frame = pack(name, Y, U, V)
    ref = cv2.cvtColor(frame, code_of(name))
    got = conv(layout, frame, h, w)
    assert np.array_equal(got, ref), (name, int((got != ref).any(-1).sum()))


@pytest.mark.parametrize("name", LAYOUTS)
def test_random_sizes_match_cv2(conv, name):
    """Even sizes from 2 x 2 up, widths that are not multiples of 4 or 16 among them (and odd heights of 4:2:2, which cv2
    converts too)."""
    layout = CODES[name][0]
    rng = np.random.default_rng(layout)
    sizes = [(2, 2), (2, 6), (4, 18), (6, 34), (720, 1280), (46, 258), (16, 514)]
    sizes += [(2 * int(rng.integers(1, 60)), 2 * int(rng.integers(1, 300))) for _ in range(20)]
    if layout > nat.YUV_NV21:
        sizes += [(1, 2), (3, 10), (17, 66)]
    for h, w in sizes:
        frame = rng.integers(0, 256, yuv.frame_shape(layout, h, w), dtype=np.uint8)
        got = conv(layout, frame, h, w)
        assert np.array_equal(got, cv2.cvtColor(frame, code_of(name))), (name, h, w)


def test_layout_of_every_alias():
    for name, (layout, aliases) in CODES.items():
        for a in aliases:
            assert yuv.layout_of(getattr(cv2, a)) == layout, a
            assert yuv.layout_of(np.int32(getattr(cv2, a))) == layout, a


@pytest.mark.parametrize("code", [cv2.COLOR_YUV2BGR, cv2.COLOR_YUV2BGRA_I420, cv2.COLOR_YUV2BGRA_NV12, cv2.COLOR_YUV2BGRA_YUY2,
                                  cv2.COLOR_YUV2RGB_I420, cv2.COLOR_YUV2RGB_NV12, cv2.COLOR_YUV2RGB_YUY2, cv2.COLOR_YUV2GRAY_420,
                                  cv2.COLOR_BGR2YUV_I420, cv2.COLOR_BGR2RGB, -1, 1000, None, "NV12", 91.0, True])
def test_other_codes_raise(code):
    with pytest.raises(ValueError):
        yuv.layout_of(code)
    with pytest.raises(ValueError):
        posenet.yuv_to_bgr_batch(np.zeros((1, 6, 4), np.uint8), code)


def test_sizes_and_shapes_cv2_rejects_raise():
    nv12, yuy2 = cv2.COLOR_YUV2BGR_NV12, cv2.COLOR_YUV2BGR_YUY2
    for shape, code in [((1, 6, 5), nv12), ((1, 7, 4), nv12), ((1, 10, 4), nv12), ((1, 6, 4, 2), nv12), ((1, 24), nv12),
                        ((1, 4, 5, 2), yuy2), ((1, 4, 4, 3), yuy2), ((1, 4, 4), yuy2), ((1, 0, 4, 2), yuy2), ((1, 3, 0), nv12)]:
        frame = np.zeros(shape, np.uint8)
        with pytest.raises(cv2.error):
            cv2.cvtColor(frame[0], code)
        with pytest.raises(ValueError):
            posenet.yuv_to_bgr_batch(frame, code)
    with pytest.raises(ValueError):
        posenet.yuv_to_bgr_batch(np.zeros((1, 6, 4), np.int16), nv12)
    for layout in range(7):
        with pytest.raises(ValueError):
            yuv.frame_shape(layout, 4, 5)
        with pytest.raises(ValueError):
            yuv.frame_shape(layout, 0, 4)
    assert yuv.frame_shape(nat.YUV_I420, 720, 1280) == (1080, 1280)
    assert yuv.frame_shape(nat.YUV_UYVY, 5, 8) == (5, 8, 2)
    with pytest.raises(ValueError):
        yuv.frame_shape(nat.YUV_NV12, 5, 8)


def test_pipeline_rejects_yuv_with_jpeg_mixed_and_odd_sizes():
    """Checked before anything touches the model or the device."""
    for kw in (dict(jpeg=True), dict(mixed=True)):
        with pytest.raises(ValueError):
            posenet.BatchPipeline(None, 2, 720, 1280, yuv=cv2.COLOR_YUV2BGR_NV12, **kw)
    for code, h, w in ((cv2.COLOR_YUV2BGR_NV12, 721, 1280), (cv2.COLOR_YUV2BGR_I420, 720, 1281), (cv2.COLOR_YUV2BGR_YUY2, 720, 1281)):
        with pytest.raises(ValueError):
            posenet.BatchPipeline(None, 2, h, w, yuv=code)
    with pytest.raises(ValueError):
        posenet.BatchPipeline(None, 2, 720, 1280, yuv=cv2.COLOR_YUV2BGRA_NV12)
