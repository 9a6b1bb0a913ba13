"""The JPEG encode arithmetic (csrc/jpeg_encode.cuh) against cv2.imencode, on the host.

The header is compiled into a small host library: a serial driver (colour, downsampling, FDCT, quantisation and dummy blocks per
block, then the entropy coder with stuffing, restart markers and headers) over the same functions csrc/jpeg_enc.cu runs in
parallel.  Its files are compared with cv2.imencode(".jpg") byte for byte.  The parallel decomposition is covered by
tests/test_gpu_jpeg_encode.py."""
import ctypes as C
import os
import subprocess

import cv2
import numpy as np
import pytest

from oracle import synth
from posenet import _native as nat
from posenet import jpeg as pj
from jpeg_corpus import corpus

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "posenet-pytorch_b200", "csrc")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")

SHIM = r"""
#include <vector>
#include "jpeg_encode.cuh"
using namespace pn::jpege;

namespace {
struct ByteSink {                      // emit_bits / flush_bits of jchuff.c: MSB first, 0xFF -> 0xFF 0x00
    std::vector<uint8_t> &o;
    uint64_t acc = 0;
    int n = 0;
    void operator()(uint32_t code, int size) {
        acc = (acc << size) | code;
        n += size;
        while (n >= 8) {
            const uint8_t b = (uint8_t)(acc >> (n - 8));
            o.push_back(b);
            if (b == 0xFF) o.push_back(0);
            n -= 8;
        }
    }
    void flush() { if (n) (*this)((1u << (8 - n)) - 1u, 8 - n); }
};
}

extern "C" {
// Serial encode of a BGR frame (rows of w * 3 bytes).  Returns the file's length, -1 for a bad sampling, -2 when cap is short.
long long t_encode(const uint8_t *frame, int h, int w, int quality, int sampling, int rst, uint8_t *out, long long cap) {
    Geom g;
    if (!geometry(h, w, sampling, rst, &g)) return -1;
    if (g.nblk == 0) return 0;
    Tables T;
    make_tables(quality, &T);
    std::vector<int16_t> coef(g.nblk * 64);
    for (long long blk = 0; blk < g.nblk; ++blk) {
        int c, bx, by, mx, sx, sy;
        block_place(g, blk, &c, &bx, &by, &mx);
        int16_t *zz = &coef[blk * 64];
        const Recip *q = T.quant[c ? 1 : 0];
        if (dummy_source(g, c, bx, by, mx, &sx, &sy)) {
            int sum = 0;
            for (int y = 0; y < 8; ++y)
                for (int x = 0; x < 8; ++x) sum += sample(g, frame, c, sx * 8 + x, sy * 8 + y) - 128;
            for (int k = 0; k < 64; ++k) zz[k] = 0;
            zz[0] = (int16_t)quantize(sum, q[0]);
            continue;
        }
        int d[64];
        for (int y = 0; y < 8; ++y)
            for (int x = 0; x < 8; ++x) d[y * 8 + x] = sample(g, frame, c, bx * 8 + x, by * 8 + y) - 128;
        for (int r = 0; r < 8; ++r) fdct_pass(d + 8 * r, 1, 0);
        for (int k = 0; k < 8; ++k) fdct_pass(d + k, 8, 1);
        for (int k = 0; k < 64; ++k) zz[zigzag_of(k)] = (int16_t)quantize(d[k], q[k]);
    }
    std::vector<uint8_t> o(kMaxHeader);
    int sof;
    o.resize(write_header(T, sampling, rst, h, w, o.data(), &sof));
    ByteSink sink{o};
    const long long per = rst > 0 ? (long long)rst * g.bpm : g.nblk;
    for (long long blk = 0; blk < g.nblk; ++blk) {
        if (blk && blk % per == 0) {
            sink.flush();
            o.push_back(0xFF);
            o.push_back((uint8_t)(0xD0 + ((blk / per - 1) & 7)));
        }
        int c, bx, by, mx;
        block_place(g, blk, &c, &bx, &by, &mx);
        const long long p = dc_pred_block(g, blk);
        const int diff = coef[blk * 64] - (p >= 0 ? coef[p * 64] : 0);
        encode_block(&coef[blk * 64], diff, T.dc[c ? 1 : 0], T.ac[c ? 1 : 0], sink);
    }
    sink.flush();
    o.push_back(0xFF);
    o.push_back(0xD9);
    if ((long long)o.size() > cap) return -2;
    memcpy(out, o.data(), o.size());
    return (long long)o.size();
}

long long t_bound(int h, int w, int quality, int sampling, int rst) {
    Geom g;
    if (!geometry(h, w, sampling, rst, &g)) return -1;
    Tables T;
    make_tables(quality, &T);
    uint8_t hdr[kMaxHeader];
    int sof;
    return encode_bound(g, write_header(T, sampling, rst, h, w, hdr, &sof));
}

// quantize() against rounding division for every |x| <= xmax and every divisor 8 * q the tables of quality 1..100 produce
// (all q in 1..255).  Returns the number of mismatches.
long long t_quant_exhaustive(int xmax) {
    long long bad = 0;
    for (int q = 1; q <= 255; ++q) {
        const int d = 8 * q;
        const Recip r = compute_reciprocal(d);
        for (int x = -xmax; x <= xmax; ++x) {
            const int a = x < 0 ? -x : x, want = (a + d / 2) / d;
            bad += quantize(x, r) != (x < 0 ? -want : want);
        }
    }
    return bad;
}
}
"""


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    d = tmp_path_factory.mktemp("jpege")
    src, lib = d / "jpege_shim.cu", d / "libjpege_shim.so"
    src.write_text(SHIM)
    cmd = [NVCC, "-O2", "-std=c++17", "-shared", "-Xcompiler", "-fPIC", "-gencode", "arch=compute_100a,code=sm_100a",
           "-I", CSRC, str(src), "-o", str(lib)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    L = C.CDLL(str(lib))
    L.t_encode.restype = C.c_longlong
    L.t_encode.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_longlong]
    L.t_bound.restype = C.c_longlong
    L.t_bound.argtypes = [C.c_int] * 5
    L.t_quant_exhaustive.restype = C.c_longlong
    L.t_quant_exhaustive.argtypes = [C.c_int]
    return L


def _opts(params):
    p = dict(zip(params[::2], params[1::2]))
    return (p.get(cv2.IMWRITE_JPEG_QUALITY, 95), p.get(cv2.IMWRITE_JPEG_SAMPLING_FACTOR, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420),
            p.get(cv2.IMWRITE_JPEG_RST_INTERVAL, 0))


def serial_encode(L, img, params):
    img = np.ascontiguousarray(img)
    q, s, rst = _opts(params)
    h, w = img.shape[:2]
    cap = max(L.t_bound(h, w, q, s, rst), 1)
    out = np.zeros(cap, np.uint8)
    n = L.t_encode(img.ctypes.data, h, w, q, s, rst, out.ctypes.data, cap)
    assert n >= 0, n
    return out[:n].tobytes()


def _colour_corpus():
    for img, params, tag in corpus(seed=5):
        if img.ndim == 3 and cv2.IMWRITE_JPEG_OPTIMIZE not in params[::2]:
            yield img, params, tag


def _check(L, img, params, tag):
    ref = cv2.imencode(".jpg", img, params)[1].tobytes()
    got = serial_encode(L, img, params)
    if got != ref:
        i = next((k for k in range(min(len(got), len(ref))) if got[k] != ref[k]), min(len(got), len(ref)))
        pytest.fail("%s: %d vs %d bytes, first difference at byte %d" % (tag, len(got), len(ref), i))


def test_corpus_byte_exact_with_cv2(shim):
    n = 0
    for img, params, tag in _colour_corpus():
        _check(shim, img, params, tag)
        n += 1
    assert n >= 100


SAMPLINGS = [cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420,
             cv2.IMWRITE_JPEG_SAMPLING_FACTOR_440, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411]


@pytest.mark.parametrize("q", [0, 1, 10, 75, 95])
def test_qualities(shim, q):
    img = synth.smooth_image(37, 61, seed=q)
    for s in SAMPLINGS:
        _check(shim, img, [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, s], "q%d s%x" % (q, s))
    _check(shim, img, [cv2.IMWRITE_JPEG_QUALITY, q], "q%d default" % q)


@pytest.mark.parametrize("hw", [(8, 8), (16, 16), (17, 33), (1, 2), (2, 1), (257, 257), (513, 513)])
def test_sizes(shim, hw):
    rng = np.random.default_rng(hw[0] * 1000 + hw[1])
    smooth = synth.smooth_image(*hw, seed=7)
    noisy = rng.integers(0, 256, hw + (3,), dtype=np.uint8)
    for s in SAMPLINGS:
        for img, tag in ((smooth, "smooth"), (noisy, "noisy")):
            _check(shim, img, [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, s], "%s %s s%x" % (hw, tag, s))


def test_extreme_content(shim):
    rng = np.random.default_rng(11)
    cases = [(np.zeros((40, 24, 3), np.uint8), "zeros"), (np.full((40, 24, 3), 255, np.uint8), "255")]
    sat = np.zeros((48, 40, 3), np.uint8)
    for k, col in enumerate([(255, 0, 0), (0, 255, 0), (0, 0, 255), (255, 255, 0), (0, 255, 255), (255, 0, 255)]):
        sat[k * 8:(k + 1) * 8] = col
    cases.append((sat, "saturated"))
    checker = (np.indices((64, 64)).sum(0) % 2 * 255).astype(np.uint8)[..., None].repeat(3, 2)
    cases.append((checker, "checker"))
    for img, tag in cases:
        for s in SAMPLINGS:
            for q in (1, 50, 100):
                _check(shim, img, [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, s], "%s q%d s%x" % (tag, q, s))
    noise = rng.integers(0, 256, (513, 513, 3), dtype=np.uint8)          # the most 0xFF stuffing
    _check(shim, noise, [cv2.IMWRITE_JPEG_QUALITY, 100, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444],
           "noise q100 444")


def test_restart_intervals(shim):
    img = synth.smooth_image(70, 45, seed=3)
    for rst in (1, 2, 7, 9, 100):
        for s in SAMPLINGS:
            _check(shim, img, [cv2.IMWRITE_JPEG_RST_INTERVAL, rst, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, s], "rst%d s%x" % (rst, s))


def test_drawn_overlays(shim):
    import posenet
    from posenet.constants import NUM_KEYPOINTS
    rng = np.random.default_rng(4)
    for h, w in ((257, 257), (200, 333)):
        img = synth.smooth_image(h, w, seed=h)
        kc = rng.uniform(-10, max(h, w) + 10, (3, NUM_KEYPOINTS, 2))
        drawn = posenet.draw_skel_and_kp(img, np.array([0.9, 0.8, 0.7]), rng.uniform(0.3, 1, (3, NUM_KEYPOINTS)), kc,
                                         min_pose_score=0.25, min_part_score=0.25)
        for q in (75, 95):
            _check(shim, drawn, [cv2.IMWRITE_JPEG_QUALITY, q], "overlay %dx%d q%d" % (h, w, q))


def test_quantiser_matches_rounding_division(shim):
    """jpeg_fdct_islow outputs are within +-8 * 1024 (the DC is the sum of 64 samples in -128..127); every divisor 8 * q of
    quality 1..100 (q in 1..255) is checked over twice that range."""
    assert shim.t_quant_exhaustive(16384) == 0


def test_bound_covers_every_file(shim):
    for img, params, tag in _colour_corpus():
        q, s, rst = _opts(params)
        n = len(cv2.imencode(".jpg", img, params)[1])
        assert n <= shim.t_bound(img.shape[0], img.shape[1], q, s, rst), tag


def test_output_parses_as_supported(shim):
    for img, params, tag in _colour_corpus():
        d = pj.parse(serial_encode(shim, img, params))
        assert d.kind == nat.JPEG_SUPPORTED, (tag, d.why)


def test_imencode_batch_rejects_unsupported_params():
    frames = np.zeros((1, 8, 8, 3), np.uint8)
    for params in ([cv2.IMWRITE_JPEG_OPTIMIZE, 1], [cv2.IMWRITE_JPEG_PROGRESSIVE, 1], [cv2.IMWRITE_JPEG_LUMA_QUALITY, 50],
                   [cv2.IMWRITE_JPEG_CHROMA_QUALITY, 50], [cv2.IMWRITE_PNG_COMPRESSION, 3], [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, 0x331111],
                   [cv2.IMWRITE_JPEG_QUALITY]):
        with pytest.raises(ValueError):
            pj.encode_options(params)
    assert pj.encode_options([cv2.IMWRITE_JPEG_OPTIMIZE, 0, cv2.IMWRITE_JPEG_PROGRESSIVE, 0]) == (95, 0x221111, 0)
    assert pj.encode_options([cv2.IMWRITE_JPEG_QUALITY, 120, cv2.IMWRITE_JPEG_RST_INTERVAL, 3]) == (100, 0x221111, 3)
    with pytest.raises(ValueError):
        pj.imencode_batch(frames, [cv2.IMWRITE_JPEG_PROGRESSIVE, 1])
