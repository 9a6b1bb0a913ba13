"""Reduced-size JPEG decode (csrc/jpeg_decode.cuh at 1/2, 1/4, 1/8) against cv2.imdecode(IMREAD_REDUCED_COLOR_d), on the host.

The header is compiled into a serial host decoder like tests/test_jpeg_cpu.py does: entropy decode and DC sums as at full size,
then the scaled IDCT of every component (jidctred.c), the scaled upsampling rule and colour conversion.  Its frames are compared
with cv2's byte for byte over the seeded corpus, a noisy q95 4:4:4 file and sizes whose downsampled widths are 1-3 at each
scale; the output size is compared with cv2's over a few hundred random (h, w, sampling, scale)."""
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

SHIM = r"""
#include <vector>
#include "jpeg_decode.cuh"
using namespace pn::jpeg;

extern "C" {
// Output size at 1 / denom, and per component (ssize, hr, vr, dw, dh, up).  Returns 0, or -1 when scaled_geometry refuses.
int t_geometry(const pn_jpeg_desc *dp, int denom, int *out) {
    Scaled g;
    if (!scaled_geometry(*dp, denom, &g)) return -1;
    out[0] = g.h;
    out[1] = g.w;
    for (int c = 0; c < 3; ++c) {
        const CompScale &s = g.comp[c];
        const int v[6] = {s.ssize, s.hr, s.vr, s.dw, s.dh, s.up};
        for (int k = 0; k < 6; ++k) out[2 + 6 * c + k] = v[k];
    }
    return 0;
}

// Serial decode of a PN_JPEG_SUPPORTED file at 1 / denom into out (ceil(h / denom) * ceil(w / denom) * 3 BGR).
int t_decode_scaled(const uint8_t *f, long long n, const pn_jpeg_desc *dp, int denom, uint8_t *out) {
    const pn_jpeg_desc &d = *dp;
    Scaled g;
    if (!scaled_geometry(d, denom, &g)) return PN_JPEG_ERR_DESC;
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
    for (int y = 0; y < g.h; ++y)
        for (int x = 0; x < g.w; ++x) pixel_bgr(d, g, pl, pitch, y, x, out + ((size_t)y * g.w + x) * 3);
    return 0;
}
}
"""


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    d = tmp_path_factory.mktemp("jpeg_reduced")
    src, lib = d / "jpeg_reduced_shim.cu", d / "libjpeg_reduced_shim.so"
    src.write_text(SHIM)
    cmd = [NVCC, "-O2", "-std=c++17", "-shared", "-Xcompiler", "-fPIC", "-gencode", "arch=compute_100a,code=sm_100a",
           "-I", CSRC, str(src), "-o", str(lib)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    L = C.CDLL(str(lib))
    L.t_geometry.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    L.t_decode_scaled.argtypes = [C.c_void_p, C.c_longlong, C.c_void_p, C.c_int, C.c_void_p]
    return L


def geometry(L, desc, denom):
    out = (C.c_int * 20)()
    assert L.t_geometry(C.addressof(desc), denom, out) == 0
    return out[0], out[1], [tuple(out[2 + 6 * c:8 + 6 * c]) for c in range(3)]


def serial_decode(L, buf, denom):
    desc = pj.parse(buf)
    assert desc.kind == nat.JPEG_SUPPORTED, (desc.kind, desc.why)
    h, w, _ = geometry(L, desc, denom)
    out = np.zeros((h, w, 3), np.uint8)
    a = np.frombuffer(buf, np.uint8)
    rc = L.t_decode_scaled(a.ctypes.data, len(buf), C.addressof(desc), denom, out.ctypes.data)
    return rc, out


def check(L, buf, denom, tag):
    ref = cv2.imdecode(np.frombuffer(buf, np.uint8), REDUCED[denom])
    rc, got = serial_decode(L, buf, denom)
    assert rc == 0, (tag, denom, rc)
    assert got.shape == ref.shape, (tag, denom, got.shape, ref.shape)
    assert np.array_equal(got, ref), (tag, denom, int((got != ref).sum()))


@pytest.mark.parametrize("denom", [1, 2, 4, 8])
def test_corpus_bit_exact_with_cv2_reduced(shim, denom):
    n = 0
    for img, params, tag in corpus(seed=5):
        check(shim, cv2.imencode(".jpg", img, params)[1].tobytes(), denom, tag)
        n += 1
    assert n >= 100


@pytest.mark.parametrize("denom", [2, 4, 8])
def test_noisy_444_q95_reduced(shim, denom):
    rng = np.random.default_rng(3)
    img = rng.integers(0, 256, (513, 513, 3), dtype=np.uint8)
    enc = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, 95, cv2.IMWRITE_JPEG_SAMPLING_FACTOR,
                                     cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444])[1].tobytes()
    check(shim, enc, denom, "noisy 444 q95")


SAMPLINGS = {"444": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444, "422": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422,
             "420": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420, "440": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_440,
             "411": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411}


@pytest.mark.parametrize("denom", [2, 4, 8])
def test_narrow_chroma_planes(shim, denom):
    """Sizes that put every component's downsampled width and height at 1, 2 and 3 samples at this scale: the edge cases of the
    fancy upsamplers (their dw > 2 condition) and of replication.  Noisy content so that every sample matters."""
    rng = np.random.default_rng(denom)
    seen = set()
    for s, f in SAMPLINGS.items():
        for w in range(1, 8 * denom + 2):
            h = int(rng.integers(1, 6 * denom))
            img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
            buf = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, 90, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, f])[1].tobytes()
            _, _, comps = geometry(shim, pj.parse(buf), denom)
            seen.update((s, c[3]) for c in comps[1:] if c[3] <= 3)
            seen.update((s, "h", c[4]) for c in comps[1:] if c[4] <= 3)
            check(shim, buf, denom, "%dx%d %s" % (h, w, s))
    for s in SAMPLINGS:
        assert {(s, 1), (s, 2), (s, 3)} <= seen, (s, sorted(x for x in seen if x[0] == s))


def test_upsampling_choice_per_scale(shim):
    """The geometry libjpeg-turbo derives (pinned by the byte comparisons above): 4:2:0 chroma needs no upsampling once the
    chroma IDCT can grow, 4:2:2 / 4:4:0 keep a fancy 2x filter until 1/8, where replication takes over."""
    img = synth.smooth_image(64, 96, 7)

    def comps(s, denom):
        buf = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, SAMPLINGS[s]])[1].tobytes()
        return geometry(shim, pj.parse(buf), denom)[2]

    FULL, H2V1, H1V2, H2V2, REP = range(5)
    assert comps("420", 1)[1][5] == H2V2 and comps("420", 2)[1][:3] == (8, 1, 1) and comps("420", 8)[1][:3] == (2, 1, 1)
    assert comps("420", 2)[0][0] == 4 and comps("420", 2)[1][5] == FULL
    assert comps("422", 2)[1][5] == H2V1 and comps("422", 4)[1][5] == H2V1 and comps("422", 8)[1][5] == REP
    assert comps("440", 4)[1][5] == H1V2 and comps("440", 8)[1][5] == REP
    assert comps("444", 8)[1] == (1, 1, 1, 12, 8, FULL)


def test_output_size_matches_cv2(shim):
    rng = np.random.default_rng(11)
    for k in range(300):
        h, w = int(rng.integers(1, 300)), int(rng.integers(1, 300))
        s = list(SAMPLINGS)[k % 5]
        denom = (2, 4, 8)[k % 3]
        buf = cv2.imencode(".jpg", np.full((h, w, 3), k % 256, np.uint8),
                           [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, SAMPLINGS[s]])[1].tobytes()
        gh, gw, _ = geometry(shim, pj.parse(buf), denom)
        ref = cv2.imdecode(np.frombuffer(buf, np.uint8), REDUCED[denom])
        assert (gh, gw) == ref.shape[:2] == (-(-h // denom), -(-w // denom)), (h, w, s, denom)


def test_gray_and_bad_scale(shim):
    g = cv2.cvtColor(synth.smooth_image(37, 61, 3), cv2.COLOR_BGR2GRAY)
    buf = cv2.imencode(".jpg", g, [cv2.IMWRITE_JPEG_QUALITY, 90])[1].tobytes()
    for denom in (2, 4, 8):
        check(shim, buf, denom, "gray")
    out = (C.c_int * 20)()
    for bad in (0, 3, 16, -2):
        assert shim.t_geometry(C.addressof(pj.parse(buf)), bad, out) == -1


# ---- the Python layer without a device: flags, ImageStream sizes and arenas ------------------------------------------------------
def test_reduce_values_are_checked():
    import posenet
    for bad in (0, 3, 16, True, "2"):
        with pytest.raises(ValueError):
            posenet.imdecode_batch([b"\xff\xd8"], reduce=bad)
        with pytest.raises(ValueError):
            posenet.ImageStream(["unused.jpg"], batch=1, height=8, width=8, reduce=bad)


@pytest.mark.parametrize("denom", [2, 8])
def test_image_stream_reduced_cv2_and_encoded(tmp_path, denom):
    """decode="cv2" yields cv2.imread(path, IMREAD_REDUCED_COLOR_d) with the reduced size taken from the first file;
    decode="gpu" parses the same files into descriptors with the reduced shapes and a full-size arena."""
    import posenet
    paths = []
    for i in range(5):
        p = tmp_path / ("f%d.jpg" % i)
        p.write_bytes(cv2.imencode(".jpg", synth.smooth_image(75, 101, 60 + i), [cv2.IMWRITE_JPEG_QUALITY, 90])[1].tobytes())
        paths.append(str(p))
    hw = (-(-75 // denom), -(-101 // denom))
    st = posenet.ImageStream(paths, batch=2, pinned=False, reduce=denom)
    assert (st.height, st.width) == hw
    got = [b.numpy()[:n].copy() for b, n in st.batches()]
    ref = np.stack([cv2.imread(p, REDUCED[denom]) for p in paths])
    assert np.array_equal(np.concatenate(got), ref)
    enc_st = posenet.ImageStream(paths, batch=2, pinned=False, reduce=denom, decode="gpu")
    assert enc_st.arena_bytes == 2 * (denom * hw[0]) * (denom * hw[1])
    for enc, n in enc_st.batches():
        assert enc.reduce == denom and enc.host_rows == [] and enc.arena.numel() == enc_st.arena_bytes
        assert enc.shapes[:n] == [hw] * n
    small = posenet.ImageStream(paths, batch=2, pinned=False, reduce=denom, decode="gpu", arena_bytes=100)
    for enc, n in small.batches():                                    # nothing fits: cv2 decodes every row at the reduced size
        assert enc.host_rows == list(range(n))
    with pytest.raises(ValueError):
        list(posenet.ImageStream(paths, batch=2, pinned=False, reduce=denom, decode="gpu", height=hw[0] + 1,
                                 width=hw[1]).batches())


def test_workspace_scaled_arguments():
    """Any scale but 1, 2, 4, 8 is an argument error; the workspace is sized for the full-size files (scale x the frames), and
    the original entry point is scale 1."""
    lib = nat.load()
    n, m = C.c_size_t(), C.c_size_t()
    for bad in (0, 3, 16, -1):
        assert lib.pn_jpeg_workspace_scaled(4, 1000, 64, 64, bad, C.byref(n)) == -1          # PN_ERR_ARG
    assert lib.pn_jpeg_workspace_scaled(4, 1000, 64, 64, 1, C.byref(n)) == 0
    assert lib.pn_jpeg_workspace(4, 1000, 64, 64, C.byref(m)) == 0 and m.value == n.value
    assert lib.pn_jpeg_workspace_scaled(4, 1000, 32, 32, 2, C.byref(m)) == 0 and m.value == n.value
    assert lib.pn_jpeg_workspace_scaled(4, 1000, 8200, 8200, 8, C.byref(m)) == -1         # a 65600-pixel file side
