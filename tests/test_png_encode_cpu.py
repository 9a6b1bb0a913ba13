"""The PNG encode arithmetic (csrc/png_encode.cuh) against cv2.imencode(".png") and Python's zlib, on the host.

The header is compiled into a small host library: a serial driver (SUB filter, the run-based Z_RLE parse, blocks of 16383
symbols, trees.c's trees and block choice, the bit writer, Adler-32, IDAT chunks with CRC-32) over the same functions
csrc/png_enc.cu runs in parallel.  Its files are compared with cv2.imencode(".png") byte for byte, and its deflate streams with
zlib.compressobj(1, DEFLATED, wbits, 8, Z_RLE) of the same bytes (the zlib cv2 loads at run time is the one Python's zlib module
uses).  The parallel decomposition is covered by tests/test_gpu_png_encode.py."""
import ctypes as C
import os
import subprocess
import zlib

import cv2
import numpy as np
import pytest

from oracle import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "posenet-pytorch_b200", "csrc")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")

SHIM = r"""
#include <string.h>
#include <vector>
#include "png_encode.cuh"
using namespace pn::pnge;

namespace {
struct ByteSink {                      // send_bits / bi_windup: LSB first
    std::vector<uint8_t> &o;
    uint32_t acc = 0;
    int n = 0;
    void operator()(uint32_t v, int len) {
        acc |= (v & ((1u << len) - 1u)) << n;
        n += len;
        while (n >= 8) {
            o.push_back((uint8_t)acc);
            acc >>= 8;
            n -= 8;
        }
    }
    void align() {
        if (n) o.push_back((uint8_t)acc);
        acc = 0;
        n = 0;
    }
};

// Serial deflate_rle + trees of data[0 .. n) into o (the deflate body only).
void deflate_body(const uint8_t *data, long long n, int wbits, std::vector<uint8_t> &o) {
    std::vector<int> lc;
    std::vector<long long> pos;
    for (long long p = 0; p < n;) {
        long long e = p + 1;
        while (e < n && data[e] == data[p]) e++;
        for (long long j = 0; j < e - p; j++) {
            int c;
            if (run_symbol_at(j, e - p, data[p], &c)) {
                lc.push_back(c);
                pos.push_back(p + j);
            }
        }
        p = e;
    }
    const long long S = (long long)lc.size(), nblk = S / kBlockSyms + 1;
    ByteSink sink{o};
    static FlushWork work;
    static BlockCode bc;
    for (long long b = 0; b < nblk; b++) {
        const long long s0 = b * kBlockSyms, s1 = s0 + kBlockSyms < S ? s0 + kBlockSyms : S;
        const bool last = b == nblk - 1;
        const long long B = s0 < S ? pos[s0] : n, E = s1 < S ? pos[s1] : n, P = last ? n : pos[s1 - 1];
        uint32_t freq[L_CODES] = {0}, matches = 0;
        for (long long s = s0; s < s1; s++) {
            if (lc[s] < 256) freq[lc[s]]++;
            else {
                freq[length_code(lc[s] - 256) + LITERALS + 1]++;
                matches++;
            }
        }
        const bool storable = B >= slides_before(P, n, wbits) << wbits;
        flush_block(freq, matches, E - B, storable, work, &bc);
        send_block_header(bc, last, sink);
        if (bc.type == STORED) {
            sink.align();
            const uint32_t len = (uint32_t)(E - B);
            sink(len & 0xFFFF, 16);
            sink(~len & 0xFFFF, 16);
            for (long long k = B; k < E; k++) o.push_back(data[k]);
        } else {
            for (long long s = s0; s < s1; s++) send_symbol(bc, lc[s], sink);
            sink(bc.code[END_BLOCK], bc.len[END_BLOCK]);
        }
    }
    sink.align();
}

uint32_t adler32(const uint8_t *d, long long n) {
    uint32_t a = 1, b = 0;
    for (long long i = 0; i < n; i++) {
        a = (a + d[i]) % kAdlerBase;
        b = (b + a) % kAdlerBase;
    }
    return b << 16 | a;
}

long long put(const std::vector<uint8_t> &o, uint8_t *out, long long cap) {
    if ((long long)o.size() > cap) return -2;
    memcpy(out, o.data(), o.size());
    return (long long)o.size();
}
}

extern "C" {
// The zlib stream deflateInit2(1, Z_DEFLATED, wbits, 8, Z_RLE) writes for data[0 .. n) given at once.
long long t_deflate(const uint8_t *data, long long n, int wbits, uint8_t *out, long long cap) {
    std::vector<uint8_t> o;
    unsigned hdr = (0x08u | (unsigned)(wbits - 8) << 4) << 8;
    hdr += 31 - hdr % 31;
    o.push_back((uint8_t)(hdr >> 8));
    o.push_back((uint8_t)hdr);
    deflate_body(data, n, wbits, o);
    uint8_t t[4];
    put_be32(t, adler32(data, n));
    o.insert(o.end(), t, t + 4);
    return put(o, out, cap);
}

// Serial PNG encode of an h x w BGR frame.
long long t_encode(const uint8_t *frame, int h, int w, uint8_t *out, long long cap) {
    if (!h || !w) return 0;
    const long long n = data_size(h, w);
    std::vector<uint8_t> f(n);
    for (long long p = 0; p < n; p++) f[p] = filtered_byte(frame, w, p);
    const int wbits = window_bits(n);
    std::vector<uint8_t> z(2);
    zlib_header(n, wbits, z.data());
    deflate_body(f.data(), n, wbits, z);
    uint8_t t[4];
    put_be32(t, adler32(f.data(), n));
    z.insert(z.end(), t, t + 4);
    std::vector<uint8_t> o(kHeadBytes);
    write_head(h, w, o.data());
    for (long long c = 0; c < (long long)z.size(); c += kIdat) {
        const long long len = (long long)z.size() - c < kIdat ? (long long)z.size() - c : kIdat;
        uint8_t hd[8];
        put_be32(hd, (uint32_t)len);
        hd[4] = 'I', hd[5] = 'D', hd[6] = 'A', hd[7] = 'T';
        o.insert(o.end(), hd, hd + 8);
        o.insert(o.end(), z.begin() + c, z.begin() + c + len);
        put_be32(t, crc32_update(crc32_update(0, hd + 4, 4), z.data() + c, len));
        o.insert(o.end(), t, t + 4);
    }
    o.resize(o.size() + kTailBytes);
    write_tail(o.data() + o.size() - kTailBytes);
    return put(o, out, cap);
}

long long t_bound(int h, int w) { return encode_bound(h, w); }
long long t_deflate_bound(long long n) { return zlib_bound(n); }
int t_window_bits(long long n) { return window_bits(n); }

// crc32_combine against the CRC of the concatenation, over split points of data[0 .. n).
int t_crc_combine(const uint8_t *d, long long n) {
    const uint32_t whole = crc32_update(0, d, n);
    for (long long k = 0; k <= n; k += 1 + k / 3)
        if (crc32_combine(crc32_update(0, d, k), crc32_update(0, d + k, n - k), n - k) != whole) return 0;
    return 1;
}
}
"""


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    d = tmp_path_factory.mktemp("pnge")
    src, lib = d / "pnge_shim.cu", d / "libpnge_shim.so"
    src.write_text(SHIM)
    cmd = [NVCC, "-O2", "-std=c++17", "-shared", "-Xcompiler", "-fPIC", "-gencode", "arch=compute_100a,code=sm_100a",
           "-I", CSRC, str(src), "-o", str(lib)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    L = C.CDLL(str(lib))
    L.t_deflate.restype = C.c_longlong
    L.t_deflate.argtypes = [C.c_void_p, C.c_longlong, C.c_int, C.c_void_p, C.c_longlong]
    L.t_encode.restype = C.c_longlong
    L.t_encode.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_longlong]
    L.t_bound.restype = C.c_longlong
    L.t_bound.argtypes = [C.c_int, C.c_int]
    L.t_deflate_bound.restype = C.c_longlong
    L.t_deflate_bound.argtypes = [C.c_longlong]
    L.t_window_bits.argtypes = [C.c_longlong]
    L.t_crc_combine.argtypes = [C.c_void_p, C.c_longlong]
    return L


def serial_encode(L, img):
    img = np.ascontiguousarray(img)
    h, w = img.shape[:2]
    cap = max(L.t_bound(h, w), 1)
    out = np.zeros(cap, np.uint8)
    n = L.t_encode(img.ctypes.data, h, w, out.ctypes.data, cap)
    assert n >= 0, "the file exceeds pn_png_encode_bound (%d)" % n
    return out[:n].tobytes()


def serial_deflate(L, data, wbits):
    a = np.frombuffer(data, np.uint8) if len(data) else np.zeros(1, np.uint8)
    cap = L.t_deflate_bound(len(data))
    out = np.zeros(cap, np.uint8)
    n = L.t_deflate(a.ctypes.data, len(data), wbits, out.ctypes.data, cap)
    assert n >= 0, "the stream exceeds the bound"
    return out[:n].tobytes()


def _check(L, img, tag):
    ref = cv2.imencode(".png", img)[1].tobytes()
    got = serial_encode(L, img)
    if got != ref:
        i = next((k for k in range(min(len(got), len(ref))) if got[k] != ref[k]), min(len(got), len(ref)))
        pytest.fail("%s: %d vs %d bytes, first difference at byte %d" % (tag, len(got), len(ref), i))


def _noise(h, w, seed, levels=256):
    rng = np.random.default_rng(seed)
    return (rng.integers(0, levels, (h, w, 3)) * (255 // max(levels - 1, 1))).astype(np.uint8)


SIZES = [(1, 1), (1, 2), (2, 3), (5, 7), (13, 40), (100, 33), (3, 2000), (513, 513), (720, 1280)]


@pytest.mark.parametrize("hw", SIZES)
def test_sizes(shim, hw):
    for tag, img in (("smooth", synth.smooth_image(*hw, seed=hw[0] + hw[1])), ("noise", _noise(*hw, seed=hw[0])),
                     ("quantised", _noise(*hw, seed=hw[1], levels=3))):
        _check(shim, img, "%s %s" % (hw, tag))


def _window_sizes():
    """(h, w) on both sides of every windowBits step and of the 16 KB threshold: the filtered size h * (3 w + 1) just at and
    just past the sizes where libpng halves the window or optimize_cmf rewrites the CMF byte."""
    out = []
    for edge in [2 ** k - 262 for k in range(8, 15)] + [2 ** k for k in range(7, 15)] + [16384]:
        for n in (edge - 1, edge, edge + 1):
            for w in range(1, 200):
                if n > 0 and n % (3 * w + 1) == 0:
                    out.append((n // (3 * w + 1), w))
                    break
    return sorted(set(out))


def test_window_bits(shim):
    sizes = _window_sizes()
    assert {shim.t_window_bits(h * (3 * w + 1)) for h, w in sizes} == set(range(9, 16))
    headers = set()
    for k, (h, w) in enumerate(sizes):
        for tag, img in (("smooth", synth.smooth_image(h, w, seed=k)), ("noise", _noise(h, w, seed=k))):
            _check(shim, img, "%dx%d %s" % (h, w, tag))
            headers.add(serial_encode(shim, img)[41:43])
    assert {b[0] >> 4 for b in headers} == set(range(0, 8))       # CMF window sizes 2^8 .. 2^15


def test_constant_frames(shim):
    for h, w in ((1, 1), (7, 300), (513, 513), (720, 1280)):
        for v in (0, 1, 255, 128):
            _check(shim, np.full((h, w, 3), v, np.uint8), "constant %d %dx%d" % (v, h, w))
    _check(shim, np.tile(np.array([3, 3, 200], np.uint8), (400, 600, 1)), "constant colour")


def test_blocky_and_striped(shim):
    rng = np.random.default_rng(9)
    img = np.kron(rng.integers(0, 256, (13, 17, 3)), np.ones((40, 60, 1))).astype(np.uint8)
    _check(shim, img, "blocky 520x1020")
    stripes = np.zeros((300, 700, 3), np.uint8)
    stripes[::2] = 255
    _check(shim, stripes, "stripes")
    half = _noise(400, 500, seed=4)
    half[:, 250:] = 17
    _check(shim, half, "half noise")


def test_drawn_overlays(shim):
    import posenet
    from posenet.constants import NUM_KEYPOINTS
    rng = np.random.default_rng(4)
    for h, w in ((257, 257), (200, 333), (513, 513)):
        img = synth.smooth_image(h, w, seed=h)
        kc = rng.uniform(-10, max(h, w) + 10, (3, NUM_KEYPOINTS, 2))
        drawn = posenet.draw_skel_and_kp(img, np.array([0.9, 0.8, 0.7]), rng.uniform(0.3, 1, (3, NUM_KEYPOINTS)), kc,
                                         min_pose_score=0.25, min_part_score=0.25)
        _check(shim, drawn, "overlay %dx%d" % (h, w))


def _unfilter(f, h, w):
    """The BGR frame whose SUB-filtered bytes are f (rows of 1 + 3 w bytes, filter byte 1)."""
    rows = f.reshape(h, 3 * w + 1)[:, 1:].reshape(h, w, 3).astype(np.int64)
    return (np.cumsum(rows, axis=1) % 256).astype(np.uint8)[..., ::-1].copy()


def test_symbol_count_multiple_of_block(shim):
    """Filtered bytes with no two equal neighbours but one run of four: 2 * 16384 bytes code as exactly 2 * 16383 symbols,
    so the stream ends with an empty final block."""
    rng = np.random.default_rng(12)
    h, w = 2, 5461
    n = h * (3 * w + 1)
    f = rng.integers(2, 256, n).astype(np.uint8)
    f[100:104] = 7
    f[::3 * w + 1] = 1
    for p in range(1, n):
        while f[p] == f[p - 1] and not 100 < p < 104 and p % (3 * w + 1):
            f[p] = rng.integers(2, 256)
    img = _unfilter(f, h, w)
    assert np.array_equal(_filtered(img), f)
    assert _count_symbols(f) == 2 * 16383
    _check(shim, img, "symbols = 2 * 16383")


def _filtered(img):
    h, w = img.shape[:2]
    rgb = img[..., ::-1].reshape(h, -1).astype(np.int16)
    f = rgb.copy()
    f[:, 3:] = rgb[:, 3:] - rgb[:, :-3]
    return np.concatenate([np.full((h, 1), 1 if w > 1 else 0, np.int16), f], axis=1).astype(np.uint8).reshape(-1)


def _count_symbols(f):
    starts = np.flatnonzero(np.concatenate([[True], f[1:] != f[:-1]]))
    lens = np.diff(np.concatenate([starts, [f.size]]))
    q, r = (lens - 1) // 258, (lens - 1) % 258
    return int((1 + q + np.where(r >= 3, 1, r)).sum())


def _streams(seed):
    rng = np.random.default_rng(seed)
    kind = seed % 5
    n = int(rng.integers(0, 3 ** int(rng.integers(1, 12))))
    if kind == 0:
        return rng.integers(0, 256, n, dtype=np.uint8).tobytes()
    if kind == 1:
        return rng.integers(0, 3, n, dtype=np.uint8).tobytes()
    if kind == 2:                                                  # runs of random lengths
        vals = rng.integers(0, 4, max(n // 8, 1), dtype=np.uint8)
        return np.repeat(vals, rng.integers(1, 600, vals.size)).tobytes()[:n]
    if kind == 3:
        return bytes(n)
    a = rng.integers(0, 256, n, dtype=np.uint8)                    # noise with long runs dropped in
    for _ in range(int(rng.integers(0, 6))):
        if n:
            p = int(rng.integers(0, n))
            a[p:p + int(rng.integers(1, 5000))] = rng.integers(0, 256)
    return a.tobytes()


def test_deflate_against_zlib(shim):
    n = 0
    for seed in range(300):
        data = _streams(seed)
        for wbits in (9, 12, 15) if len(data) > 1000 else (15,):
            c = zlib.compressobj(1, zlib.DEFLATED, wbits, 8, zlib.Z_RLE)
            ref = c.compress(data) + c.flush()
            got = serial_deflate(shim, data, wbits)
            assert got == ref, "seed %d, %d bytes, wbits %d" % (seed, len(data), wbits)
            assert len(got) <= shim.t_deflate_bound(len(data))
            n += 1
    assert n > 300


def test_deflate_block_edges(shim):
    """Inputs around one and two blocks of 16383 symbols, literal-only and with long runs, in small windows (stored blocks
    whose start has slid out of the window are coded instead)."""
    rng = np.random.default_rng(3)
    base = bytes(np.arange(200000) % 251 * 7 % 256 ^ rng.integers(0, 2, 200000).astype(np.int64) << 7)
    for n in (16382, 16383, 16384, 32766, 32767, 49149, 100000):
        data = base[:n]
        for wbits in (9, 10, 13, 15):
            c = zlib.compressobj(1, zlib.DEFLATED, wbits, 8, zlib.Z_RLE)
            assert serial_deflate(shim, data, wbits) == c.compress(data) + c.flush(), (n, wbits)
    runs = bytes(200000)
    for wbits in (9, 15):
        c = zlib.compressobj(1, zlib.DEFLATED, wbits, 8, zlib.Z_RLE)
        assert serial_deflate(shim, runs, wbits) == c.compress(runs) + c.flush()


def test_crc32_combine(shim):
    rng = np.random.default_rng(5)
    a = rng.integers(0, 256, 3000, dtype=np.uint8)
    assert shim.t_crc_combine(a.ctypes.data, a.size) == 1


def test_bound_covers_every_file(shim):
    cases = [(hw, _noise(*hw, seed=1)) for hw in SIZES] + [((64, 64), np.zeros((64, 64, 3), np.uint8))]
    for (h, w), img in cases:
        assert len(cv2.imencode(".png", img)[1]) <= shim.t_bound(h, w), (h, w)


def test_params_are_rejected():
    from posenet import png as pp
    for params in ([cv2.IMWRITE_PNG_COMPRESSION, 1], [cv2.IMWRITE_PNG_COMPRESSION, 3], [cv2.IMWRITE_PNG_STRATEGY, 3],
                   [cv2.IMWRITE_PNG_BILEVEL, 0], [cv2.IMWRITE_PNG_FILTER, 1], [cv2.IMWRITE_JPEG_QUALITY, 95],
                   [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, 0x221111], [cv2.IMWRITE_PNG_COMPRESSION]):
        with pytest.raises(ValueError):
            pp.encode_options(params)
    if hasattr(cv2, "IMWRITE_PNG_ZLIBBUFFER_SIZE"):
        with pytest.raises(ValueError):
            pp.encode_options([cv2.IMWRITE_PNG_ZLIBBUFFER_SIZE, 8192])
    pp.encode_options([])
    pp.encode_options(())
    import posenet
    with pytest.raises(ValueError):
        posenet.imencode_png_batch(np.zeros((1, 8, 8, 3), np.uint8), [cv2.IMWRITE_PNG_COMPRESSION, 1])
