"""EXIF orientation on the JPEG path, on the host: pn_jpeg_parse_oriented's acceptance rule and the orientation map of
csrc/jpeg_decode.cuh against cv2.imdecode, which rotates a file after decoding it (at the reduced size too).

The header is compiled into a serial host decoder as tests/test_jpeg_reduced_cpu.py does, plus the output-to-source pixel map the
colour kernel applies.  Its frames are compared with cv2's byte for byte for every orientation, sampling and scale.  A seeded
fuzz of Exif segments checks that whatever the oriented parser accepts, cv2 rotates the same way, and that the default parser
sends every file cv2 might rotate to the host."""
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
REDUCED = {1: cv2.IMREAD_COLOR, 2: cv2.IMREAD_REDUCED_COLOR_2, 4: cv2.IMREAD_REDUCED_COLOR_4, 8: cv2.IMREAD_REDUCED_COLOR_8}
SAMPLINGS = (cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420,
             cv2.IMWRITE_JPEG_SAMPLING_FACTOR_440, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411)

SHIM = r"""
#include <vector>
#include "jpeg_decode.cuh"
using namespace pn::jpeg;

extern "C" {
// Oriented output size of a descriptor at 1 / denom.
void t_oriented_size(const pn_jpeg_desc *dp, int denom, int *hw) {
    oriented_size(dp->orientation, (dp->height + denom - 1) / denom, (dp->width + denom - 1) / denom, &hw[0], &hw[1]);
}

// Serial decode of a PN_JPEG_SUPPORTED file at 1 / denom, written through the orientation map into out (the oriented frame).
int t_decode_oriented(const uint8_t *f, long long n, const pn_jpeg_desc *dp, int denom, uint8_t *out) {
    const pn_jpeg_desc &d = *dp;
    Scaled g;
    if (!scaled_geometry(d, denom, &g) || d.orientation > 8) return PN_JPEG_ERR_DESC;
    std::vector<uint8_t> ds;
    std::vector<uint32_t> seg{0};
    bool end = false;
    for (long long q = d.scan_offset; q < n && !end; ++q) {
        const int prev = q > d.scan_offset ? f[q - 1] : -1, next = q + 1 < n ? f[q + 1] : -1;
        switch (classify_byte(prev, f[q], next)) {
        case BYTE_DATA: ds.push_back(f[q]); break;
        case BYTE_RST: seg.push_back((uint32_t)ds.size()); break;
        case BYTE_END: end = true; break;
        default: break;
        }
    }
    if (!end || (int)seg.size() != d.n_segments) return PN_JPEG_ERR_RESTART;
    seg.push_back((uint32_t)ds.size());
    const long long mcus = (long long)d.mcus_x * d.mcus_y, nblk = mcus * d.blocks_per_mcu;
    std::vector<int16_t> coef(nblk * 64);
    long long gi = 0;
    for (int s = 0; s < d.n_segments; ++s) {
        const BitSrc src{ds.data() + seg[s], seg[s + 1] - seg[s]};
        const long long m = mcus - (long long)s * d.restart_interval < d.restart_interval ? mcus - (long long)s * d.restart_interval
                                                                                           : d.restart_interval;
        State st{0, 0, 0};
        unsigned last_dc[3] = {0, 0, 0};
        for (long long b = 0; b < m * d.blocks_per_mcu; ++b, ++gi) {
            const int c = d.mcu_comp[st.b];
            if (!decode_block(d, src, st, &coef[gi * 64])) return PN_JPEG_ERR_CODE;
            last_dc[c] += (unsigned)(int)coef[gi * 64];
            coef[gi * 64] = (int16_t)(uint16_t)last_dc[c];
        }
    }
    std::vector<uint8_t> planes[3];
    int pitch[3] = {0, 0, 0};
    for (int c = 0; c < d.ncomp; ++c) {
        pitch[c] = d.comp[c].bw * g.comp[c].ssize;
        planes[c].assign((size_t)pitch[c] * d.comp[c].bh * g.comp[c].ssize, 0);
    }
    for (gi = 0; gi < nblk; ++gi) {
        int c, bx, by, ws[64];
        block_place(d, gi, &c, &bx, &by);
        const int ss = g.comp[c].ssize;
        for (int k = 0; k < 8; ++k) idct_column_scaled(&coef[gi * 64], d.quant[c], ss, k, ws);
        for (int r = 0; r < ss; ++r)
            idct_row_scaled(&coef[gi * 64], d.quant[c], ws, ss, r, &planes[c][((size_t)by * ss + r) * pitch[c] + (size_t)bx * ss]);
    }
    const uint8_t *pl[3] = {planes[0].data(), d.ncomp > 1 ? planes[1].data() : nullptr, d.ncomp > 1 ? planes[2].data() : nullptr};
    int OH, OW;
    oriented_size(d.orientation, g.h, g.w, &OH, &OW);
    for (int y = 0; y < OH; ++y)
        for (int x = 0; x < OW; ++x) {
            int sy, sx;
            orient_source(d.orientation, g.h, g.w, y, x, &sy, &sx);
            pixel_bgr(d, g, pl, pitch, sy, sx, out + ((size_t)y * OW + x) * 3);
        }
    return 0;
}
}
"""


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    d = tmp_path_factory.mktemp("jpeg_orient")
    src, lib = d / "jpeg_orient_shim.cu", d / "libjpeg_orient_shim.so"
    src.write_text(SHIM)
    cmd = [NVCC, "-O2", "-std=c++17", "-shared", "-Xcompiler", "-fPIC", "-gencode", "arch=compute_100a,code=sm_100a",
           "-I", CSRC, str(src), "-o", str(lib)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    L = C.CDLL(str(lib))
    L.t_oriented_size.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    L.t_decode_oriented.argtypes = [C.c_void_p, C.c_longlong, C.c_void_p, C.c_int, C.c_void_p]
    return L


# ---- Exif segments --------------------------------------------------------------------------------------------------------------
def tiff(entries, le=False, magic=42, ifd=8, count=None, order=None):
    """A TIFF header + IFD0 with ``entries`` of (tag, type, count, value); ``count`` overrides the entry count written."""
    order = order if order is not None else (b"II" if le else b"MM")

    def u16(v):
        return int(v & 0xFFFF).to_bytes(2, "little" if le else "big")

    def u32(v):
        return int(v & 0xFFFFFFFF).to_bytes(4, "little" if le else "big")
    body = order + u16(magic) + u32(ifd) + bytes(max(ifd - 8, 0))
    body += u16(len(entries) if count is None else count)
    for tag, typ, cnt, val in entries:
        value = u16(val) + b"\0\0" if typ == 3 else u32(val)
        body += u16(tag) + u16(typ) + u32(cnt) + value
    return body + b"\0\0\0\0"


def app1(payload):
    return b"\xff\xe1" + (len(payload) + 2).to_bytes(2, "big") + payload


def exif(o, le=False):
    return app1(b"Exif\0\0" + tiff([(0x0112, 3, 1, o)], le=le))


def with_segments(base, *segments):
    return base[:2] + b"".join(segments) + base[2:]


def orient_np(r, o):
    """cv2's applyExifOrientation as numpy views (the table in include/posenet_b200.h)."""
    return {1: r, 2: r[:, ::-1], 3: r[::-1, ::-1], 4: r[::-1], 5: r.transpose(1, 0, 2), 6: r[::-1].transpose(1, 0, 2),
            7: r[::-1, ::-1].transpose(1, 0, 2), 8: r[:, ::-1].transpose(1, 0, 2)}.get(o, r)


def decode(buf, flag=cv2.IMREAD_COLOR):
    return cv2.imdecode(np.frombuffer(buf, np.uint8), flag)


def serial_decode(L, buf, denom):
    d = pj.parse(buf, orientation="gpu")
    assert d.kind == nat.JPEG_SUPPORTED, (d.kind, d.why)
    hw = (C.c_int * 2)()
    L.t_oriented_size(C.addressof(d), denom, hw)
    out = np.zeros((hw[0], hw[1], 3), np.uint8)
    a = np.frombuffer(buf, np.uint8)
    assert L.t_decode_oriented(a.ctypes.data, len(buf), C.addressof(d), denom, out.ctypes.data) == 0
    assert pj.frame_size(d, denom) == (hw[0], hw[1])
    return d, out


# ---- the orientation map against cv2 ---------------------------------------------------------------------------------------------
SIZES = ((1, 1), (1, 19), (23, 1), (7, 5), (16, 48), (17, 33), (37, 61), (45, 30))


@pytest.mark.parametrize("denom", [1, 2, 4, 8])
def test_every_orientation_sampling_and_scale_bit_exact(shim, denom):
    rng = np.random.default_rng(denom)
    n = 0
    for h, w in SIZES:
        for si, samp in enumerate(SAMPLINGS):
            img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8) if (h + si) % 2 else synth.smooth_image(h, w, h * 31 + si)
            base = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, 90, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, samp])[1].tobytes()
            for o in range(1, 9):
                buf = with_segments(base, exif(o, le=(o + si) % 2 == 1))
                d, got = serial_decode(shim, buf, denom)
                assert d.orientation == (o if o > 1 else 0)
                ref = decode(buf, REDUCED[denom])
                assert got.shape == ref.shape, (h, w, si, o, got.shape, ref.shape)
                assert np.array_equal(got, ref), (h, w, si, o, denom, int((got != ref).sum()))
                n += 1
    assert n == len(SIZES) * 5 * 8


def test_gray_and_restart_intervals_rotated(shim):
    g = cv2.cvtColor(synth.smooth_image(29, 53, 4), cv2.COLOR_BGR2GRAY)
    gray = cv2.imencode(".jpg", g, [cv2.IMWRITE_JPEG_QUALITY, 90])[1].tobytes()
    rst = cv2.imencode(".jpg", synth.smooth_image(70, 45, 5), [cv2.IMWRITE_JPEG_RST_INTERVAL, 3])[1].tobytes()
    for base in (gray, rst):
        for o in (3, 6, 7):
            for denom in (1, 4):
                buf = with_segments(base, exif(o))
                assert np.array_equal(serial_decode(shim, buf, denom)[1], decode(buf, REDUCED[denom]))


# ---- the acceptance rule ---------------------------------------------------------------------------------------------------------
XMP = app1(b"http://ns.adobe.com/xap/1.0/\0<x:xmpmeta xmlns:x='adobe:ns:meta/'/>")


TYPE_BYTES = {1: 1, 2: 1, 3: 2, 4: 4, 5: 8, 7: 1, 9: 4, 10: 8}


def random_segment(rng):
    """One APP1 Exif segment with random variations, whether it is well formed with one orientation entry (SHORT, count 1, value
    1..8) that cv2 reaches -- the entries ahead of it in TIFF order, of known types, their data inside the segment -- or without
    one, and the orientation value (None without the entry)."""
    le = bool(rng.integers(2))
    fine = True
    order = None
    if rng.random() < 0.08:
        order, fine = [b"IM", b"XX", b"ii", b"MI"][int(rng.integers(4))], False
    magic = 42
    if rng.random() < 0.06:
        magic, fine = [43, 0, 0x2A00][int(rng.integers(3))], False
    ifd = 8 if rng.random() < 0.8 else int(rng.integers(9, 20))
    entries = []
    for _ in range(int(rng.integers(0, 4))):
        typ = int(rng.choice([1, 2, 3, 4, 5, 7, 0, 13]))
        cnt = int(rng.choice([1, 2, 3, 4, 6, 12, 40, 1000]))
        val = int(rng.integers(0, 64)) if rng.random() < 0.7 else int(rng.integers(0, 1 << 16))
        entries.append((int(rng.choice([0x0100, 0x010E, 0x010F, 0x0110, 0x011A, 0x0128, 0x8769])), typ, cnt, val))
    value, at = None, None
    if rng.random() < 0.8:
        typ = 3 if rng.random() < 0.85 else int(rng.choice([1, 4, 9]))
        cnt = 1 if rng.random() < 0.85 else int(rng.choice([0, 2, 4]))
        val = int(rng.integers(1, 9)) if rng.random() < 0.85 else int(rng.choice([0, 9, 255, 65535]))
        at = int(rng.integers(len(entries) + 1))
        entries.insert(at, (0x0112, typ, cnt, val))
        if typ == 3 and cnt == 1 and 1 <= val <= 8:
            value = val
        else:
            fine = False
        if rng.random() < 0.05:                                   # a second orientation entry in the same IFD
            entries.append((0x0112, 3, 1, int(rng.integers(1, 9))))
            fine = False
    tail = bytes(int(rng.integers(0, 48)))                        # room for entries' data
    body = tiff(entries, le=le, magic=magic, ifd=ifd, order=order) + tail
    for tag, typ, cnt, val in entries[:at]:                       # what cv2 reads ahead of the orientation entry
        n = TYPE_BYTES.get(typ, 0) * cnt
        off = val << 16 if typ == 3 and not le else val           # a SHORT's value sits in the first two bytes of the field
        if not (tag < 0x0112 and typ in TYPE_BYTES and (n <= 4 or off + n <= len(body))):
            fine = False
    if rng.random() < 0.08:                                       # an IFD count larger or smaller than the entries present
        k = len(entries) + int(rng.integers(1, 4)) if rng.random() < 0.6 else int(rng.integers(0, max(len(entries), 1)))
        body = body[:ifd] + int(k).to_bytes(2, "little" if le else "big") + body[ifd + 2:]
        fine = False
    if rng.random() < 0.04:                                       # an IFD offset inside the header or past the segment
        body = body[:4] + int(rng.choice([0, 4, 7, 5000])).to_bytes(4, "little" if le else "big") + body[8:]
        fine = False
    body = b"Exif\0\0" + body
    if rng.random() < 0.06:
        body, fine = body[:int(rng.integers(6, len(body)))], False
    return app1(body), fine, value


def test_exif_fuzz_oriented_parser_agrees_with_cv2():
    """Whatever pn_jpeg_parse_oriented accepts with orientation o, cv2 decodes as the unrotated frame under o; every well-formed
    single-segment file is accepted.  pn_jpeg_parse accepts only files cv2 leaves unrotated, with the same descriptor."""
    rng = np.random.default_rng(2024)
    img = rng.integers(0, 256, (5, 7, 3), dtype=np.uint8)
    base = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, 90])[1].tobytes()
    plain = decode(base)
    stats = dict(accepted=0, rotated=0, host=0, multi_accepted=0)
    for k in range(3000):
        segs, fines, values = [], [], []
        for _ in range(1 if rng.random() < 0.6 else int(rng.integers(2, 4))):
            s, f, v = random_segment(rng)
            segs.append(s)
            fines.append(f)
            values.append(v)
        pre = []
        if rng.random() < 0.15:
            pre.append(XMP)
        if rng.random() < 0.05:
            pre.append(app1(b"NotExif\0" + bytes(10)))
        buf = with_segments(base, *(pre + segs))
        ref = decode(buf)
        assert ref is not None
        dg, dc = pj.parse(buf, orientation="gpu"), pj.parse(buf)
        if dg.kind == nat.JPEG_SUPPORTED:
            o = dg.orientation or 1
            assert np.array_equal(ref, orient_np(plain, o)), (k, o, buf[:80])
            stats["accepted"] += 1
            stats["rotated"] += o > 1
            stats["multi_accepted"] += len(segs) > 1
        else:
            assert dg.why == dc.why
            stats["host"] += 1
        if dc.kind == nat.JPEG_SUPPORTED:
            assert dc.orientation == 0 and np.array_equal(ref, plain), k
            assert bytes(dc) == bytes(dg), k                         # identical descriptors for unrotated files
        if len(segs) == 1 and fines[0]:
            assert dg.kind == nat.JPEG_SUPPORTED, (k, values, dg.why)
            assert dg.orientation == (values[0] if values[0] and values[0] > 1 else 0)
    assert stats["rotated"] > 300 and stats["host"] > 1000 and stats["multi_accepted"] > 50, stats


def test_default_parse_sends_every_rotating_segment_to_the_host():
    """cv2 takes the first Exif segment with a readable orientation: 6 followed by 1, or by a segment without the tag, is rotated.
    pn_jpeg_parse used to keep the last segment's value and decoded such files unrotated on the GPU."""
    img = synth.smooth_image(40, 56, seed=2)
    base = cv2.imencode(".jpg", img)[1].tobytes()
    plain = decode(base)
    no_tag = app1(b"Exif\0\0" + tiff([(0x010F, 2, 4, 0)]))
    rotated = [(exif(6), exif(1)), (exif(6), no_tag), (no_tag, exif(6)), (exif(6, le=True), exif(1, le=True))]
    for segs in rotated:
        buf = with_segments(base, *segs)
        assert np.array_equal(decode(buf), orient_np(plain, 6))
        d = pj.parse(buf)
        assert (d.kind, d.why) == (nat.JPEG_HOST, nat.JPEG_WHY["exif_orientation"]), segs
    # 1 then 6: cv2 keeps the frame, but the segments disagree -- the host decodes it either way
    buf = with_segments(base, exif(1), exif(6))
    assert np.array_equal(decode(buf), plain)
    assert pj.parse(buf).kind == nat.JPEG_HOST and pj.parse(buf, orientation="gpu").kind == nat.JPEG_HOST
    # the oriented parse takes agreeing segments, and segments without the tag, and refuses disagreeing ones
    assert pj.parse(with_segments(base, exif(6), no_tag), orientation="gpu").orientation == 6
    assert pj.parse(with_segments(base, no_tag, exif(8), exif(8, le=True)), orientation="gpu").orientation == 8
    assert pj.parse(with_segments(base, exif(6), exif(1)), orientation="gpu").why == nat.JPEG_WHY["exif_orientation"]
    # several segments that all say 1 or nothing stay supported and unrotated
    for segs in ((exif(1), exif(1)), (no_tag, exif(1)), (no_tag, no_tag)):
        d = pj.parse(with_segments(base, *segs))
        assert d.kind == nat.JPEG_SUPPORTED and d.orientation == 0


def test_lenient_cases_stay_on_the_host():
    """Orientation entries cv2 reads more loosely than pn_jpeg_parse_oriented (LONG, count 2, out-of-range values, an IFD count
    larger than the entries present) keep today's classification in both parsers."""
    base = cv2.imencode(".jpg", synth.smooth_image(24, 40, seed=3))[1].tobytes()
    for t in (tiff([(0x0112, 4, 1, 6)]), tiff([(0x0112, 3, 2, 6)]), tiff([(0x0112, 3, 1, 9)]), tiff([(0x0112, 3, 1, 0)]),
              tiff([(0x0112, 3, 1, 6)], count=3), tiff([(0x0112, 3, 1, 6)], order=b"XX")):
        buf = with_segments(base, app1(b"Exif\0\0" + t))
        for orientation in ("cv2", "gpu"):
            d = pj.parse(buf, orientation=orientation)
            assert (d.kind, d.why) == (nat.JPEG_HOST, nat.JPEG_WHY["exif_orientation"]), t


def test_default_parse_unchanged_on_the_corpus():
    """Files without an orientation get the same descriptor from both parsers, with orientation 0; a single Exif segment keeps
    its classification."""
    for img, params, tag in corpus(seed=5):
        buf = cv2.imencode(".jpg", img, params)[1].tobytes()
        a, b = pj.parse(buf), pj.parse(buf, orientation="gpu")
        assert a.kind == nat.JPEG_SUPPORTED and a.orientation == 0 and bytes(a) == bytes(b), tag
        one = with_segments(buf, exif(1))
        assert bytes(pj.parse(one)) == bytes(pj.parse(one, orientation="gpu")), tag
        six = with_segments(buf, exif(6))
        assert pj.parse(six).why == nat.JPEG_WHY["exif_orientation"]
        d = pj.parse(six, orientation="gpu")
        assert d.kind == nat.JPEG_SUPPORTED and d.orientation == 6 and pj.frame_size(d, 1) == (d.width, d.height), tag


# ---- the Python layer and the workspace without a device ----------------------------------------------------------------------
def test_orientation_option_is_checked():
    import posenet
    buf = cv2.imencode(".jpg", synth.smooth_image(8, 8, 1))[1].tobytes()
    for bad in ("GPU", None, 1, "host"):
        with pytest.raises(ValueError):
            pj.parse(buf, orientation=bad)
        with pytest.raises(ValueError):
            posenet.imdecode_batch([buf], orientation=bad)
    with pytest.raises(ValueError):
        posenet.ImageStream(["unused.jpg"], batch=1, height=8, width=8, orientation="gpu")        # decode="cv2"
    with pytest.raises(ValueError):
        posenet.ImageStream(["unused.jpg"], batch=1, height=8, width=8, decode="gpu", orientation="yes")


def test_image_stream_oriented_shapes(tmp_path):
    """decode="gpu", orientation="gpu": rotated files are parsed into descriptors with their rotated, reduced shapes; a dense
    stream refuses a portrait among landscapes as the cv2 stream does, a mixed one takes both."""
    import posenet
    base = cv2.imencode(".jpg", synth.smooth_image(75, 101, 3), [cv2.IMWRITE_JPEG_QUALITY, 90])[1].tobytes()
    paths = []
    for i, o in enumerate((1, 6, 3, 8, 1)):
        p = tmp_path / ("f%d.jpg" % i)
        p.write_bytes(with_segments(base, exif(o)))
        paths.append(str(p))
    for denom in (1, 4):
        h, w = pj.reduced_size(75, 101, denom)
        side = max(h, w)
        st = posenet.ImageStream(paths, batch=5, height=side, width=side, mixed=True, pinned=False, decode="gpu", reduce=denom,
                                 orientation="gpu")
        ref = posenet.ImageStream(paths, batch=5, height=side, width=side, mixed=True, pinned=False, reduce=denom)
        (enc, n, shapes), = list(st.batches())
        (_, _, ref_shapes), = list(ref.batches())
        assert enc.host_rows == [] and shapes == ref_shapes == [(h, w), (w, h), (h, w), (w, h), (h, w)]
        old = posenet.ImageStream(paths, batch=5, height=side, width=side, mixed=True, pinned=False, decode="gpu", reduce=denom)
        (enc, _, shapes), = list(old.batches())
        assert enc.host_rows == [1, 2, 3] and shapes == ref_shapes
    for kw in (dict(decode="gpu", orientation="gpu"), dict()):
        with pytest.raises(ValueError):
            list(posenet.ImageStream(paths, batch=5, height=75, width=101, pinned=False, **kw).batches())


def test_workspace_holds_either_order():
    """A rotated file that fits max_h x max_w is stored as max_w x max_h: the workspace is the same for both orders."""
    lib = nat.load()
    a, b = C.c_size_t(), C.c_size_t()
    for h, w, d in ((64, 200, 1), (3024, 4032, 1), (756, 1008, 4), (1, 65500, 1)):
        assert lib.pn_jpeg_workspace_scaled(8, 1 << 20, h, w, d, C.byref(a)) == 0
        assert lib.pn_jpeg_workspace_scaled(8, 1 << 20, w, h, d, C.byref(b)) == 0
        assert a.value == b.value, (h, w, d)
