"""Progressive JPEG decode (csrc/jpeg_progressive.cuh + pn_jpeg_parse_progressive) against cv2.imdecode, on the host.

jpeg_progressive.cuh is compiled with the baseline decode headers into a serial host decoder, as tests/test_jpeg_cpu.py does: it
decodes every restart segment of every scan of the parser's scan table, in a given scan order, then runs the baseline IDCT,
upsampling and colour conversion.  Its frames are compared with cv2's byte for byte over cv2's progressive files (the seeded
corpus, a quality sweep, reduce 2 / 4 / 8), over files whose independent scans were permuted and whose DHT segments were moved,
and the parser's classifications (incomplete scripts, patched progressions, libjpeg warnings) are checked against cv2."""
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
PROG = [cv2.IMWRITE_JPEG_PROGRESSIVE, 1]

SHIM = r"""
#include <vector>
#include "jpeg_progressive.cuh"
using namespace pn::jpeg;

extern "C" {
// Serial decode at 1 / denom into out (ceil(h / denom) * ceil(w / denom) * 3 BGR): the scans order[0 .. n_scans) of the table
// (scans, huff), each cut at its RST markers, then the baseline IDCT / upsampling / colour.  Returns 0 or a status < 0.
int t_decode(const uint8_t *f, long long n, const pn_jpeg_desc *dp, const pn_jpeg_scan *scans, int n_scans,
             const pn_jpeg_huff *huff, const int *order, int denom, uint8_t *out) {
    const pn_jpeg_desc &d = *dp;
    Scaled g;
    if (!scaled_geometry(d, denom, &g)) return PN_JPEG_ERR_DESC;
    const long long nblk = (long long)d.mcus_x * d.mcus_y * d.blocks_per_mcu;
    std::vector<int16_t> coef(nblk * 64, 0);
    for (int o = 0; o < n_scans; ++o) {
        const pn_jpeg_scan &S = scans[order[o]];
        const long long units = scan_units(d, S), nseg = scan_segments(d, S);
        const long long ri = S.restart_interval > 0 ? S.restart_interval : units;
        long long p = S.start;
        for (long long k = 0; k < nseg; ++k) {
            long long e = S.end;
            if (k + 1 < nseg) {
                e = next_restart(f, p, S.end);
                if (e == S.end || f[e + 1] != 0xD0 + (k & 7)) return PN_JPEG_ERR_RESTART;
            }
            const long long u0 = k * ri;
            const int st = decode_scan_segment(d, S, huff, f, p, e, u0, units - u0 < ri ? units - u0 : ri, coef.data());
            if (st) return st;
            p = e + 2;
        }
    }
    std::vector<uint8_t> planes[3];
    int pitch[3] = {0, 0, 0};
    for (int c = 0; c < d.ncomp; ++c) {
        pitch[c] = d.comp[c].bw * g.comp[c].ssize;
        planes[c].assign((size_t)pitch[c] * d.comp[c].bh * g.comp[c].ssize, 0);
    }
    for (long long gi = 0; gi < nblk; ++gi) {
        int c, bx, by, ws[64];
        block_place(d, gi, &c, &bx, &by);
        const int ss = g.comp[c].ssize;
        for (int k = 0; k < 8; ++k) idct_column_scaled(&coef[gi * 64], d.quant[c], ss, k, ws);
        for (int r = 0; r < ss; ++r)
            idct_row_scaled(&coef[gi * 64], d.quant[c], ws, ss, r, &planes[c][((size_t)by * ss + r) * pitch[c] + (size_t)bx * ss]);
    }
    const uint8_t *pl[3] = {planes[0].data(), d.ncomp > 1 ? planes[1].data() : nullptr, d.ncomp > 1 ? planes[2].data() : nullptr};
    for (int y = 0; y < g.h; ++y)
        for (int x = 0; x < g.w; ++x) pixel_bgr(d, g, pl, pitch, y, x, out + ((size_t)y * g.w + x) * 3);
    return 0;
}
}
"""


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    d = tmp_path_factory.mktemp("jpeg_progressive")
    src, lib = d / "jpeg_progressive_shim.cu", d / "libjpeg_progressive_shim.so"
    src.write_text(SHIM)
    cmd = [NVCC, "-O2", "-std=c++17", "-shared", "-Xcompiler", "-fPIC", "-gencode", "arch=compute_100a,code=sm_100a",
           "-I", CSRC, str(src), "-o", str(lib)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    L = C.CDLL(str(lib))
    L.t_decode.argtypes = [C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    return L


def table_parts(table):
    """(scans, huff bytes) of a scan table."""
    h = nat.JpegScans.from_buffer_copy(table)
    at = C.sizeof(nat.JpegScans)
    scans = [nat.JpegScan.from_buffer_copy(table, at + i * C.sizeof(nat.JpegScan)) for i in range(h.n_scans)]
    return scans, table[at + h.n_scans * C.sizeof(nat.JpegScan):]


def serial_decode(L, buf, desc, scans, huff, denom=1, order=None):
    h, w = pj.reduced_size(desc.height, desc.width, denom)
    out = np.zeros((h, w, 3), np.uint8)
    a = np.frombuffer(buf, np.uint8)
    sc = (nat.JpegScan * len(scans))(*scans)
    hb = np.frombuffer(huff, np.uint8).copy() if huff else np.zeros(1, np.uint8)
    order = np.arange(len(scans), dtype=np.int32) if order is None else np.asarray(order, np.int32)
    rc = L.t_decode(a.ctypes.data, len(buf), C.addressof(desc), C.addressof(sc), len(scans), hb.ctypes.data, order.ctypes.data,
                    denom, out.ctypes.data)
    return rc, out


def check(L, buf, denom, tag):
    desc, table = pj.parse(buf, progressive="gpu")
    assert desc.kind == nat.JPEG_SUPPORTED_PROGRESSIVE, (tag, desc.kind, desc.why)
    scans, huff = table_parts(table)
    rc, got = serial_decode(L, buf, desc, scans, huff, denom)
    ref = cv2.imdecode(np.frombuffer(buf, np.uint8), REDUCED[denom])
    assert rc == 0, (tag, denom, rc)
    assert got.shape == ref.shape and np.array_equal(got, ref), (tag, denom, int((got != ref).sum()))
    return desc, scans


# ---- bit-exact decode ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("denom", [1, 2, 4, 8])
def test_corpus_bit_exact_with_cv2(shim, denom):
    """The seeded corpus (five samplings and grayscale, q50 / 90 / 100, 1x1 to 720x1280, restart intervals 1 and 7, smooth and
    noisy content) encoded progressive by cv2."""
    n = 0
    for img, params, tag in corpus(seed=7):
        check(shim, cv2.imencode(".jpg", img, params + PROG)[1].tobytes(), denom, tag)
        n += 1
    assert n >= 100


def test_quality_sweep(shim):
    rng = np.random.default_rng(4)
    samp = [cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422]
    for q in range(1, 101):
        h, w = int(rng.integers(1, 60)), int(rng.integers(1, 60))
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8) if q % 2 else synth.smooth_image(h, w, seed=q)
        params = [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, samp[q % 3]] + PROG
        if q % 5 == 0:
            params += [cv2.IMWRITE_JPEG_RST_INTERVAL, 1 + q % 7]
        check(shim, cv2.imencode(".jpg", img, params)[1].tobytes(), 1, "q%d %dx%d" % (q, h, w))


def test_simple_progression_waves(shim):
    """jpeg_simple_progression in colour is three waves: the first scans of disjoint bands, their refinements, the last luma
    refinement; grayscale has the same depth."""
    img = synth.smooth_image(45, 70, seed=1)
    _, scans = check(shim, cv2.imencode(".jpg", img, PROG)[1].tobytes(), 1, "colour")
    assert [s.wave for s in scans] == [0, 0, 0, 0, 0, 1, 1, 1, 1, 2]
    g = cv2.cvtColor(img, cv2.COLOR_BGR2GRAY)
    _, scans = check(shim, cv2.imencode(".jpg", g, PROG)[1].tobytes(), 1, "gray")
    assert max(s.wave for s in scans) == 2


# ---- rewritten files: scans permuted within a wave, DHT segments moved ----------------------------------------------------------
def segments(buf):
    """The file as (marker, bytes) pieces: every marker segment, each SOS with its entropy-coded data, EOI."""
    out, p = [], 2
    while True:
        m = buf[p + 1]
        if m == 0xD9:
            out.append((m, buf[p:p + 2]))
            return buf[:2], out
        ln = (buf[p + 2] << 8) | buf[p + 3]
        end = p + 2 + ln
        if m == 0xDA:
            while not (buf[end] == 0xFF and buf[end + 1] not in (0x00, 0xFF) and not 0xD0 <= buf[end + 1] <= 0xD7):
                end += 1
        out.append((m, buf[p:end]))
        p = end


def rewrite(buf, rng):
    """The same image with the scans of each wave in a random order (DC scans ahead of AC scans), every scan taking the DHT segments that preceded it, each
    DHT split into one segment per table in reverse order; the DHT ahead of the first scan moves in front of the DQT."""
    soi, segs = segments(buf)
    head, groups, cur = [], [], []
    for m, b in segs:
        if m == 0xD9:
            break
        if m == 0xDA:
            groups.append(cur + [(m, b)])
            cur = []
        elif groups or m == 0xC4:
            cur.append((m, b))
        else:
            head.append((m, b))
    desc, table = pj.parse(buf, progressive="gpu")
    scans = table_parts(table)[0]
    waves = [s.wave for s in scans]
    order = []
    for w in range(max(waves) + 1):          # a component's AC scans stay behind its first DC scan (libjpeg warns otherwise)
        for dc in (True, False):
            order += list(rng.permutation([i for i, s in enumerate(scans) if s.wave == w and (s.ss == 0) == dc]))

    def split_dht(b):
        body, o, parts = b[4:], 0, []
        while o < len(body):
            n = 17 + sum(body[o + 1:o + 17])
            t = body[o:o + n]
            parts.append(b"\xff\xc4" + (len(t) + 2).to_bytes(2, "big") + t)
            o += n
        return b"".join(reversed(parts))

    out = [soi]
    first = [b for m, b in groups[order[0]] if m == 0xC4]
    dqt_at = next(i for i, (m, _) in enumerate(head) if m == 0xDB)
    for i, (m, b) in enumerate(head):
        if i == dqt_at:
            out += [split_dht(x) for x in first]
        out.append(b)
    for k, gi in enumerate(order):
        for m, b in groups[gi]:
            if m == 0xC4 and k == 0:
                continue
            out.append(split_dht(b) if m == 0xC4 else b)
    out.append(b"\xff\xd9")
    return b"".join(out), [waves[i] for i in order]


def test_permuted_scans_and_moved_tables(shim):
    rng = np.random.default_rng(12)
    samp = [cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411]
    n = 0
    for k in range(12):
        h, w = int(rng.integers(8, 200)), int(rng.integers(8, 200))
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8) if k % 2 else synth.smooth_image(h, w, seed=k)
        if k % 4 == 3:
            img = cv2.cvtColor(img, cv2.COLOR_BGR2GRAY)
        params = [cv2.IMWRITE_JPEG_QUALITY, 40 + 5 * k, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, samp[k % 3]] + PROG
        if k % 3 == 2:
            params += [cv2.IMWRITE_JPEG_RST_INTERVAL, 3]
        buf = cv2.imencode(".jpg", img, params)[1].tobytes()
        ref = cv2.imdecode(np.frombuffer(buf, np.uint8), cv2.IMREAD_COLOR)
        new, waves = rewrite(buf, rng)
        assert new != buf
        assert np.array_equal(cv2.imdecode(np.frombuffer(new, np.uint8), cv2.IMREAD_COLOR), ref)   # the same image to cv2
        _, scans = check(shim, new, 1, "rewritten %d" % k)
        assert [s.wave for s in scans] == waves
        # the serial decoder in any order that keeps the waves
        order = sorted(range(len(scans)), key=lambda i: (scans[i].wave, rng.random()))
        desc, table = pj.parse(new, progressive="gpu")
        sc, huff = table_parts(table)
        rc, got = serial_decode(shim, new, desc, sc, huff, 1, order)
        assert rc == 0 and np.array_equal(got, ref)
        n += 1
    assert n == 12


# ---- classifications -------------------------------------------------------------------------------------------------------------
def test_incomplete_scripts_are_host_and_cv2_smooths_them(shim):
    """Dropping trailing scans leaves coefficients unrefined: the file is the host's.  cv2 decodes such a file with block smoothing,
    unlike a decode of the remaining scans as they are (the complete file's table cut short), which is why the rule matters."""
    img = synth.smooth_image(96, 128, seed=3)
    buf = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, 85] + PROG)[1].tobytes()
    desc, table = pj.parse(buf, progressive="gpu")
    scans, huff = table_parts(table)
    differs = 0
    for drop in range(1, len(scans)):
        cut = buf[:scans[-drop - 1].end] + b"\xff\xd9"
        d, t = pj.parse(cut, progressive="gpu")
        assert d.kind == nat.JPEG_HOST and d.why == nat.JPEG_WHY["progressive"] and t == b"", drop
        rc, plain = serial_decode(shim, cut, desc, scans[:-drop], huff)
        assert rc == 0
        differs += not np.array_equal(plain, cv2.imdecode(np.frombuffer(cut, np.uint8), cv2.IMREAD_COLOR))
    assert differs >= (len(scans) - 1) // 2, differs


def patch_scan(buf, index, ss=None, se=None, ah=None, al=None):
    soi, segs = segments(buf)
    out, k = [soi], 0
    for m, b in segs:
        if m == 0xDA:
            if k == index:
                b = bytearray(b)
                ns = b[4]
                o = 5 + 2 * ns
                if ss is not None:
                    b[o] = ss
                if se is not None:
                    b[o + 1] = se
                if ah is not None or al is not None:
                    b[o + 2] = ((b[o + 2] >> 4) if ah is None else ah) << 4 | ((b[o + 2] & 15) if al is None else al)
                b = bytes(b)
            k += 1
        out.append(b)
    return b"".join(out)


def test_patched_progressions_are_host():
    img = synth.smooth_image(40, 56, seed=5)
    buf = cv2.imencode(".jpg", img, PROG)[1].tobytes()
    assert pj.parse(buf, progressive="gpu")[0].kind == nat.JPEG_SUPPORTED_PROGRESSIVE
    for kw in ({"index": 0, "al": 2},            # the DC refinement's Ah no longer matches
               {"index": 0, "se": 5},            # a DC scan with Se > 0
               {"index": 1, "ss": 0},            # an AC band from 0: a one-component "DC" scan with Se 5
               {"index": 1, "se": 64},           # Se past 63
               {"index": 1, "ss": 6, "se": 5},   # Ss > Se
               {"index": 5, "ah": 3},            # Ah != Al + 1
               {"index": 5, "ah": 1, "al": 0},   # Ah other than the previous Al (2)
               {"index": 2, "al": 14}):          # Al out of range
        d, t = pj.parse(patch_scan(buf, **kw), progressive="gpu")
        assert d.kind == nat.JPEG_HOST and t == b"", kw
    # an AC scan before any DC scan of its component
    soi, segs = segments(buf)
    sos = [i for i, (m, _) in enumerate(segs) if m == 0xDA]
    moved = segs[:sos[0] - 1] + segs[sos[0] + 1:sos[1] + 1] + segs[sos[0] - 1:sos[0] + 1] + segs[sos[1] + 1:]
    d, _ = pj.parse(soi + b"".join(b for _, b in moved), progressive="gpu")
    assert d.kind == nat.JPEG_HOST


def test_parser_options_and_baseline_files():
    """Baseline files come back exactly as from pn_jpeg_parse / _oriented with no table; progressive="cv2" is the old parser;
    other values are a ValueError; a table that does not fit the caller's buffer makes the file the host's."""
    rng = np.random.default_rng(2)
    for img, params, tag in corpus(seed=8)[::7]:
        buf = cv2.imencode(".jpg", img, params)[1].tobytes()
        for orientation in ("cv2", "gpu"):
            d, t = pj.parse(buf, orientation, "gpu")
            assert bytes(d) == bytes(pj.parse(buf, orientation)) and t == b"", tag
        prog = cv2.imencode(".jpg", img, params + PROG)[1].tobytes()
        d = pj.parse(prog)
        assert d.kind == nat.JPEG_HOST and d.why == nat.JPEG_WHY["progressive"]
        cut = prog[:int(len(prog) * rng.uniform(0.2, 0.95))]
        assert pj.parse(cut, progressive="gpu")[0].kind == nat.JPEG_HOST
    for bad in ("GPU", None, 1):
        with pytest.raises(ValueError):
            pj.parse(buf, progressive=bad)
    prog = cv2.imencode(".jpg", synth.smooth_image(30, 30, seed=1), PROG)[1].tobytes()
    a = np.frombuffer(prog, np.uint8)
    _, need = pj.parse_progressive(a, "cv2", np.zeros(nat.JPEG_SCAN_TABLE_MAX, np.uint8))
    d, n = pj.parse_progressive(a, "cv2", np.zeros(need - 1, np.uint8))
    assert d.kind == nat.JPEG_HOST and n == need
    d, n = pj.parse_progressive(a, "cv2", np.zeros(need, np.uint8))
    assert d.kind == nat.JPEG_SUPPORTED_PROGRESSIVE and n == need


def test_supported_progressive_files_decode_without_warnings(tmp_path):
    """A file the progressive parser accepts is one cv2 decodes without a libjpeg warning (cv2 in a subprocess, as in
    tests/test_jpeg_cpu.py): cv2's progressive corpus, truncated copies, patched progressions and incomplete scripts."""
    rng = np.random.default_rng(10)
    files = []
    for k, (img, params, tag) in enumerate(corpus(seed=9)):
        if k % 3:
            continue
        buf = cv2.imencode(".jpg", img, params + PROG)[1].tobytes()
        kind = (k // 3) % 6
        if kind == 0:
            buf = buf[:int(len(buf) * rng.uniform(0.3, 0.95))]
        elif kind == 1:
            buf = patch_scan(buf, 0, al=2)
        elif kind == 2:
            s = table_parts(pj.parse(buf, progressive="gpu")[1])[0]
            buf = buf[:s[-2].end] + b"\xff\xd9"
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
    assert warned, "the truncated and patched files should make libjpeg warn"
    accepted = 0
    for p in files:
        if pj.parse(open(p, "rb").read(), progressive="gpu")[0].kind == nat.JPEG_SUPPORTED_PROGRESSIVE:
            assert p not in warned, p
            accepted += 1
    assert accepted >= len(files) // 3


def test_stream_progressive_option(tmp_path):
    """ImageStream(progressive="gpu") needs decode="gpu"; it packs each progressive file 8-byte aligned with its scan table after
    it and takes no more arena space than those; a file and table that do not fit go to cv2."""
    import posenet
    paths = []
    for i in range(5):
        p = tmp_path / ("f%d.jpg" % i)
        params = [cv2.IMWRITE_JPEG_QUALITY, 90] + (PROG if i % 2 == 0 else [])
        p.write_bytes(cv2.imencode(".jpg", synth.smooth_image(33, 47, 60 + i), params)[1].tobytes())
        paths.append(str(p))
    with pytest.raises(ValueError):
        posenet.ImageStream(paths, batch=2, pinned=False, progressive="gpu")
    with pytest.raises(ValueError):
        posenet.ImageStream(paths, batch=2, pinned=False, decode="gpu", progressive="yes")
    st = posenet.ImageStream(paths, batch=5, pinned=False, decode="gpu", progressive="gpu", workers=1, arena_bytes=1 << 17)
    (enc, n), = list(st.batches())
    assert enc.host_rows == [] and n == 5
    descs = [nat.JpegDesc.from_buffer_copy(enc.descs.numpy(), i * C.sizeof(nat.JpegDesc)) for i in range(5)]
    assert [d.kind for d in descs] == [2, 0, 2, 0, 2]
    end = 0
    for d in descs:
        assert d.file_offset % 8 == 0 and d.file_offset >= end
        end = d.file_offset + d.file_bytes
        if d.kind == 2:
            t = enc.arena.numpy()[pj.align8(end):].tobytes()
            h = nat.JpegScans.from_buffer_copy(t)
            assert h.n_scans == 10 and h.n_waves == 3
            end = pj.align8(end) + C.sizeof(nat.JpegScans) + h.n_scans * C.sizeof(nat.JpegScan) + h.n_huff * C.sizeof(nat.JpegHuff)
    assert enc.used == end
    cv2_st = posenet.ImageStream(paths, batch=5, pinned=False, decode="gpu")
    (enc, n), = list(cv2_st.batches())
    assert sorted(enc.host_rows) == [0, 2, 4]
    small = posenet.ImageStream(paths, batch=5, pinned=False, decode="gpu", progressive="gpu", workers=1,
                                arena_bytes=os.path.getsize(paths[0]) + 16)
    (enc, n), = list(small.batches())
    assert 0 in enc.host_rows
