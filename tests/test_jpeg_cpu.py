"""The JPEG decode arithmetic (csrc/jpeg_decode.cuh) and the header parser (pn_jpeg_parse) against cv2, on the host.

The header is compiled into a small host library: a serial driver (de-stuff, decode every restart interval block by block, DC
sums, IDCT, upsampling, colour) over the same functions csrc/jpeg.cu runs in parallel.  Its frames are compared with
cv2.imdecode(IMREAD_COLOR) byte for byte over a seeded corpus written by cv2.imencode.  The parallel decomposition (self-
synchronising subsequences) is covered by tests/test_gpu_jpeg.py."""
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
#include "jpeg_decode.cuh"
using namespace pn::jpeg;

extern "C" {
long long t_desc_size() { return sizeof(pn_jpeg_desc); }

// Serial decode of a PN_JPEG_SUPPORTED file into out (h * w * 3 BGR).  Returns 0 or a PN_JPEG_ERR_* code.
int t_decode(const uint8_t *f, long long n, const pn_jpeg_desc *dp, uint8_t *out) {
    const pn_jpeg_desc &d = *dp;
    // de-stuff, segment starts
    std::vector<uint8_t> ds;
    std::vector<uint32_t> seg{0};
    bool end = false;
    for (long long q = d.scan_offset; q < n && !end; ++q) {
        const int prev = q > d.scan_offset ? f[q - 1] : -1, next = q + 1 < n ? f[q + 1] : -1;
        switch (classify_byte(prev, f[q], next)) {
        case BYTE_DATA: ds.push_back(f[q]); break;
        case BYTE_RST:
            if (next - 0xD0 != (int)((seg.size() - 1) & 7)) return PN_JPEG_ERR_RESTART;
            seg.push_back((uint32_t)ds.size());
            break;
        case BYTE_END: end = true; break;
        default: break;
        }
    }
    if (!end) return PN_JPEG_ERR_NO_END;
    if ((int)seg.size() != d.n_segments) return PN_JPEG_ERR_RESTART;
    seg.push_back((uint32_t)ds.size());
    const long long mcus = (long long)d.mcus_x * d.mcus_y, nblk = mcus * d.blocks_per_mcu;
    std::vector<int16_t> coef(nblk * 64);
    long long g = 0;
    for (int s = 0; s < d.n_segments; ++s) {
        const BitSrc src{ds.data() + seg[s], seg[s + 1] - seg[s]};
        const long long m = mcus - (long long)s * d.restart_interval < d.restart_interval ? mcus - (long long)s * d.restart_interval
                                                                                          : d.restart_interval;
        State st{0, 0, 0};
        unsigned last_dc[3] = {0, 0, 0};
        for (long long b = 0; b < m * d.blocks_per_mcu; ++b, ++g) {
            const int c = d.mcu_comp[st.b];
            if (!decode_block(d, src, st, &coef[g * 64])) return PN_JPEG_ERR_CODE;
            last_dc[c] += (unsigned)(int)coef[g * 64];
            coef[g * 64] = (int16_t)(uint16_t)last_dc[c];
        }
        const uint32_t bits = (seg[s + 1] - seg[s]) * 8u;
        if (st.pos > bits || bits - st.pos > 7) return PN_JPEG_ERR_LENGTH;
    }
    std::vector<uint8_t> planes[3];
    int pitch[3];
    for (int c = 0; c < d.ncomp; ++c) {
        pitch[c] = d.comp[c].bw * 8;
        planes[c].assign((size_t)pitch[c] * d.comp[c].bh * 8, 0);
    }
    for (g = 0; g < nblk; ++g) {
        int c, bx, by, ws[64];
        block_place(d, g, &c, &bx, &by);
        for (int k = 0; k < 8; ++k) idct_column(&coef[g * 64], d.quant[c], k, ws);
        for (int r = 0; r < 8; ++r) idct_row(ws, r, &planes[c][((size_t)by * 8 + r) * pitch[c] + bx * 8]);
    }
    const uint8_t *pl[3] = {planes[0].data(), d.ncomp > 1 ? planes[1].data() : nullptr, d.ncomp > 1 ? planes[2].data() : nullptr};
    for (int y = 0; y < d.height; ++y)
        for (int x = 0; x < d.width; ++x) pixel_bgr(d, pl, pitch, y, x, out + ((size_t)y * d.width + x) * 3);
    return 0;
}

// The parallel decomposition of csrc/jpeg.cu run serially: speculative exits, merge points, the chain walk (with its serial
// fallback), and every subsequence's entry recomputed from the nearest chain element.  out: [subsequences, entries that differ
// from the true decoder state, subsequences the walk followed serially, deepest recompute (subsequences), deepest merge
// continuation (subsequences)].
int t_decompose(const uint8_t *f, long long n, const pn_jpeg_desc *dp, int S, int limit, long long *out) {
    const pn_jpeg_desc &d = *dp;
    std::vector<uint8_t> ds;
    std::vector<uint32_t> seg{0};
    for (long long q = d.scan_offset; q < n; ++q) {
        const int prev = q > d.scan_offset ? f[q - 1] : -1, next = q + 1 < n ? f[q + 1] : -1;
        const int k = classify_byte(prev, f[q], next);
        if (k == BYTE_DATA) ds.push_back(f[q]);
        else if (k == BYTE_RST) seg.push_back((uint32_t)ds.size());
        else if (k == BYTE_END) break;
    }
    seg.push_back((uint32_t)ds.size());
    for (int i = 0; i < 5; ++i) out[i] = 0;
    for (size_t sg = 0; sg + 1 < seg.size(); ++sg) {
        const BitSrc src{ds.data() + seg[sg], seg[sg + 1] - seg[sg]};
        const uint32_t bits = src.nbytes * 8u;
        const int nk = bits / S > 1 ? (int)(bits / S) : 1;
        out[0] += nk;
        if (nk == 1) continue;
        std::vector<uint64_t> e1(nk), truth(nk), ech(nk);
        std::vector<uint32_t> c1(nk), c2(nk), bch(nk), tb(nk);
        std::vector<int> m(nk), flag(nk, 0);
        State t{0, 0, 0};
        uint32_t cnt = 0;
        for (int k = 0; k + 1 < nk; ++k) {                       // the true states, serially
            if (!advance(d, src, t, (uint32_t)(k + 1) * S, &cnt)) return PN_JPEG_ERR_CODE;
            truth[k] = pack(t);
            tb[k] = cnt;
        }
        for (int k = 0; k + 1 < nk; ++k) {                       // spec
            State s{(uint32_t)k * S, 0, 0};
            c1[k] = 0;
            e1[k] = advance(d, src, s, (uint32_t)(k + 1) * S, &c1[k]) ? pack(s) : kBadState;
        }
        for (int k = 0; k + 1 < nk; ++k) {                       // merge
            m[k] = e1[k] == kBadState ? MERGE_NONE
                                      : merge_point(d, src, unpack(e1[k]), k, nk, S, limit, [&](int j) { return e1[j]; }, &c2[k]);
            if (m[k] >= 0 && m[k] - k > out[4]) out[4] = m[k] - k;
        }
        int c = 0;                                                  // walk
        uint32_t cum = c1[0];
        flag[0] = 1;
        bch[0] = cum;
        for (;;) {
            if (m[c] == MERGE_TAIL) break;
            if (m[c] >= 0) {
                cum += c2[c];
                c = m[c];
                flag[c] = 1;
                bch[c] = cum;
                continue;
            }
            State s = unpack(flag[c] == 2 ? ech[c] : e1[c]);
            bool merged = false;
            for (int j = c + 1; j < nk - 1 && !merged; ++j) {
                if (!advance(d, src, s, (uint32_t)(j + 1) * S, &cum)) return PN_JPEG_ERR_CODE;
                ++out[2];
                c = j;
                ech[j] = pack(s);
                bch[j] = cum;
                flag[j] = 2;
                merged = pack(s) == e1[j];
            }
            if (!merged) break;
        }
        for (int k = 1; k < nk; ++k) {                           // entries, as write_kernel computes them
            int cc = k - 1;
            while (cc > 0 && flag[cc] == 0) --cc;
            State s = unpack(flag[cc] == 2 ? ech[cc] : e1[cc]);
            uint32_t b = bch[cc];
            if (cc < k - 1) advance(d, src, s, (uint32_t)k * S, &b);
            if (k - 1 - cc > out[3]) out[3] = k - 1 - cc;
            out[1] += pack(s) != truth[k - 1] || b != tb[k - 1];
        }
    }
    return 0;
}
}
"""


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    d = tmp_path_factory.mktemp("jpeg")
    src, lib = d / "jpeg_shim.cu", d / "libjpeg_shim.so"
    src.write_text(SHIM)
    cmd = [NVCC, "-O2", "-std=c++17", "-shared", "-Xcompiler", "-fPIC", "-gencode", "arch=compute_100a,code=sm_100a",
           "-I", CSRC, str(src), "-o", str(lib)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    L = C.CDLL(str(lib))
    L.t_desc_size.restype = C.c_longlong
    L.t_decode.argtypes = [C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p]
    L.t_decompose.argtypes = [C.c_void_p, C.c_longlong, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    return L


def serial_decode(L, buf):
    desc = pj.parse(buf)
    assert desc.kind == nat.JPEG_SUPPORTED, (desc.kind, desc.why)
    out = np.zeros((desc.height, desc.width, 3), np.uint8)
    a = np.frombuffer(buf, np.uint8)
    rc = L.t_decode(a.ctypes.data, len(buf), C.addressof(desc), out.ctypes.data)
    return rc, out


def test_descriptor_layout_matches_header(shim):
    assert shim.t_desc_size() == C.sizeof(nat.JpegDesc)


def test_corpus_bit_exact_with_cv2(shim):
    checked = 0
    for img, params, tag in corpus(seed=5):
        ok, enc = cv2.imencode(".jpg", img, params)
        assert ok
        buf = enc.tobytes()
        ref = cv2.imdecode(enc, cv2.IMREAD_COLOR)
        rc, got = serial_decode(shim, buf)
        assert rc == 0, (tag, rc)
        assert np.array_equal(got, ref), (tag, int((got != ref).sum()))
        checked += 1
    assert checked >= 100


def test_noisy_444_q95_is_large_and_exact(shim):
    rng = np.random.default_rng(3)
    img = rng.integers(0, 256, (513, 513, 3), dtype=np.uint8)
    ok, enc = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, 95, cv2.IMWRITE_JPEG_SAMPLING_FACTOR,
                                         cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444])
    assert len(enc) > 0.3 * img.size                                  # ~40 % of raw: long scans, dense in stuffed bytes
    rc, got = serial_decode(shim, enc.tobytes())
    assert rc == 0 and np.array_equal(got, cv2.imdecode(enc, cv2.IMREAD_COLOR))


SUB_BITS, MERGE_LIMIT = 1024, 64                                    # csrc/jpeg.cu


def decompose(L, buf):
    desc = pj.parse(buf)
    a = np.frombuffer(buf, np.uint8)
    out = (C.c_longlong * 5)()
    assert L.t_decompose(a.ctypes.data, len(buf), C.addressof(desc), SUB_BITS, MERGE_LIMIT, out) == 0
    return dict(zip(("subsequences", "wrong_entries", "walked_serially", "recompute_depth", "merge_depth"), out))


def test_parallel_decomposition_finds_the_true_states(shim):
    """Every subsequence's entry state and first block index, as the kernels derive them from speculative exits and merge
    points, equal the serial decoder's -- over the whole corpus, restart intervals included."""
    for img, params, tag in corpus(seed=5):
        r = decompose(shim, cv2.imencode(".jpg", img, params)[1].tobytes())
        assert r["wrong_entries"] == 0, (tag, r)


@pytest.mark.parametrize("kind", ["c2", "c3", "noisy420", "noisy444"])
def test_synchronisation_depth_is_bounded(shim, kind):
    """The decode is parallel in practice, not only correct: the walk never falls back to following the true path serially,
    and no thread decodes more than a few subsequences beyond its own (smooth frames) or MERGE_LIMIT (noise at q95 4:4:4,
    which resynchronises slowest)."""
    rng = np.random.default_rng(1)
    img, params, depth = {
        "c2": (synth.smooth_image(513, 513, 3), [cv2.IMWRITE_JPEG_QUALITY, 90], 12),
        "c3": (synth.smooth_image(720, 1280, 50), [cv2.IMWRITE_JPEG_QUALITY, 90], 12),
        "noisy420": (rng.integers(0, 256, (513, 513, 3), dtype=np.uint8), [cv2.IMWRITE_JPEG_QUALITY, 90], 48),
        "noisy444": (rng.integers(0, 256, (513, 513, 3), dtype=np.uint8),
                     [cv2.IMWRITE_JPEG_QUALITY, 95, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444], 64),
    }[kind]
    r = decompose(shim, cv2.imencode(".jpg", img, params)[1].tobytes())
    assert r["subsequences"] > 300 and r["wrong_entries"] == 0, r
    assert r["walked_serially"] == 0, r
    assert r["merge_depth"] <= depth and r["recompute_depth"] <= depth, r


def _patch_sof(buf, fn):
    b = bytearray(buf)
    i = b.find(b"\xff\xc0")
    fn(b, i)
    return bytes(b)


def test_parser_classifies_host_files():
    img = synth.smooth_image(40, 56, seed=1)
    base = cv2.imencode(".jpg", img)[1].tobytes()
    assert pj.parse(base).kind == nat.JPEG_SUPPORTED
    prog = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_PROGRESSIVE, 1])[1].tobytes()
    assert (pj.parse(prog).kind, pj.parse(prog).why) == (nat.JPEG_HOST, nat.JPEG_WHY["progressive"])

    def sof9(b, i):
        b[i + 1] = 0xC9
    assert pj.parse(_patch_sof(base, sof9)).why == nat.JPEG_WHY["arithmetic"]

    def p12(b, i):
        b[i + 4] = 12
    assert pj.parse(_patch_sof(base, p12)).why == nat.JPEG_WHY["precision"]

    def four(b, i):
        b[i + 9] = 4
    assert pj.parse(_patch_sof(base, four)).why == nat.JPEG_WHY["components"]
    # EXIF APP1 with orientation 6 right after SOI (cv2.imread rotates such files)
    tiff = b"MM\x00\x2a\x00\x00\x00\x08" + b"\x00\x01" + b"\x01\x12\x00\x03\x00\x00\x00\x01\x00\x06\x00\x00" + b"\x00\x00\x00\x00"
    payload = b"Exif\x00\x00" + tiff
    app1 = b"\xff\xe1" + (len(payload) + 2).to_bytes(2, "big") + payload
    rot = base[:2] + app1 + base[2:]
    assert pj.parse(rot).why == nat.JPEG_WHY["exif_orientation"]
    assert cv2.imdecode(np.frombuffer(rot, np.uint8), cv2.IMREAD_COLOR).shape[:2] == (56, 40)
    one = base[:2] + app1.replace(b"\x00\x06\x00\x00\x00\x00\x00\x00", b"\x00\x01\x00\x00\x00\x00\x00\x00") + base[2:]
    assert pj.parse(one).kind == nat.JPEG_SUPPORTED
    # truncated: inside the headers, and inside the scan (no EOI)
    assert pj.parse(base[:100]).kind == nat.JPEG_HOST
    assert pj.parse(base[:len(base) - 40]).why == nat.JPEG_WHY["truncated"]
    assert pj.parse(b"\x89PNG\r\n\x1a\n").why == nat.JPEG_WHY["not_jpeg"]


def test_supported_files_decode_without_warnings(tmp_path):
    """A file the parser calls supported is one cv2 decodes without a libjpeg warning.  cv2 runs in a subprocess (libjpeg warns on
    stderr from C); a marker written to the same stream before each file attributes every warning to its file."""
    rng = np.random.default_rng(9)
    files = []
    for k, (img, params, tag) in enumerate(corpus(seed=6)):
        if k % 4:
            continue
        buf = cv2.imencode(".jpg", img, params)[1].tobytes()
        if k % 8 == 0:                                                     # truncated copies must not be called supported
            buf = buf[:int(len(buf) * rng.uniform(0.3, 0.95))]
        p = tmp_path / ("f%03d.jpg" % k)
        p.write_bytes(buf)
        files.append(str(p))
    code = "import os, sys, cv2\nfor p in sys.argv[1:]:\n    os.write(2, ('@@' + p + '\\n').encode())\n    cv2.imread(p)\n"
    r = subprocess.run([os.sys.executable, "-c", code] + files, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    warned, cur = set(), None
    for line in r.stderr.splitlines():
        if line.startswith("@@"):
            cur = line[2:]
        elif line.strip():
            warned.add(cur)
    assert warned, "the truncated files should make libjpeg warn"
    for p in files:
        if pj.parse(open(p, "rb").read()).kind == nat.JPEG_SUPPORTED:
            assert p not in warned, p
