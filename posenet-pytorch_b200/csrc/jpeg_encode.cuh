// Baseline JPEG encode arithmetic, restated from libjpeg-turbo 3.1 (what cv2 4.13 runs for cv2.imencode(".jpg") without
// optimised tables or progressive mode), as __host__ __device__ functions: csrc/jpeg_enc.cu runs them in parallel,
// tests/test_jpeg_encode_cpu.py compiles them into a serial host encoder and compares its files with cv2 byte for byte.
//
//   colour:        jccolor.c rgb_ycc_convert (SCALEBITS 16, ONE_HALF rounding, CBCR_OFFSET; Cb / Cr round with ONE_HALF - 1)
//   edges:         jcsample.c expand_right_edge to width_in_blocks * 8 * h_expand, jcprepct.c expand_bottom_edge to a whole
//                  MCU row: a full-resolution sample at (x, y) is the conversion of pixel (min(x, w - 1), min(y, h - 1))
//   downsampling:  h2v1 (bias 0, 1, ..), h2v2 (bias 1, 2, ..), int_downsample ((sum + n / 2) / n) for 4:4:0 and 4:1:1
//   DCT:           jpeg_fdct_islow (jfdctint.c): CONST_BITS 13, PASS1_BITS 2, on samples - 128
//   quantisation:  jcdctmgr.c quantize with compute_reciprocal's (reciprocal, correction, shift) of divisor 8 * qtbl[k]
//   dummy blocks:  jccoefct.c compress_data: MCU padding blocks are zero with the DC of the block before them in the MCU
//   entropy:       jchuff.c encode_one_block with the Annex K tables (jstdhuff.c); 0xFF stuffing, 1-bit padding, RSTn
//   headers:       jcmarker.c: SOI, APP0 (JFIF 1.01), DQT x 2, SOF0, DHT x 4, DRI, SOS
#pragma once
#include <stdint.h>

#ifdef __CUDACC__
#define PN_JEHD __host__ __device__ __forceinline__
#else
#define PN_JEHD inline
#endif

namespace pn {
namespace jpege {

// ---- geometry ------------------------------------------------------------------------------------------------------------------
// cv2's IMWRITE_JPEG_SAMPLING_FACTOR_* values: 0xHV1111, the luma sampling factors (chroma is always 1 x 1).
PN_JEHD bool luma_factors(int sampling, int *h, int *v) {
    switch (sampling) {
    case 0x411111: *h = 4; *v = 1; return true;
    case 0x221111: *h = 2; *v = 2; return true;
    case 0x211111: *h = 2; *v = 1; return true;
    case 0x121111: *h = 1; *v = 2; return true;
    case 0x111111: *h = 1; *v = 1; return true;
    default: return false;
    }
}

struct Geom {
    int h, w;                 // image size
    int hmax, vmax;           // luma sampling factors (= the maximum)
    int mcus_x, mcus_y, bpm;  // MCUs, blocks per MCU (hmax * vmax + 2)
    int bw[3], bh[3];         // width_in_blocks / height_in_blocks per component (no MCU padding)
    int rst;                  // MCUs per restart interval (0: none)
    int nseg;                 // restart intervals
    long long nblk;           // blocks in the scan (MCU padding included)
};

PN_JEHD int div_up(long long a, long long b) { return (int)((a + b - 1) / b); }

// false for an unknown sampling; a 0 x 0 image has no blocks (an empty file)
PN_JEHD bool geometry(int h, int w, int sampling, int rst, Geom *g) {
    int hm, vm;
    if (!luma_factors(sampling, &hm, &vm)) return false;
    g->h = h;
    g->w = w;
    g->hmax = hm;
    g->vmax = vm;
    g->rst = rst;
    if (h <= 0 || w <= 0) {
        g->mcus_x = g->mcus_y = 0;
        g->bpm = hm * vm + 2;
        for (int c = 0; c < 3; ++c) g->bw[c] = g->bh[c] = 0;
        g->nseg = 0;
        g->nblk = 0;
        return true;
    }
    g->mcus_x = div_up(w, 8 * hm);
    g->mcus_y = div_up(h, 8 * vm);
    g->bpm = hm * vm + 2;
    for (int c = 0; c < 3; ++c) {
        const int hc = c ? 1 : hm, vc = c ? 1 : vm;
        g->bw[c] = div_up((long long)w * hc, 8ll * hm);
        g->bh[c] = div_up((long long)h * vc, 8ll * vm);
    }
    const long long mcus = (long long)g->mcus_x * g->mcus_y;
    g->nseg = rst > 0 ? (int)((mcus + rst - 1) / rst) : 1;
    g->nblk = mcus * g->bpm;
    return true;
}

// Block g of the scan (MCU order, then the MCU's blocks: hmax x vmax luma blocks row by row, Cb, Cr): component and position.
PN_JEHD void block_place(const Geom &g, long long blk, int *comp, int *bx, int *by, int *mx) {
    const long long m = blk / g.bpm;
    const int b = (int)(blk - m * g.bpm);
    const int mcx = (int)(m % g.mcus_x), mcy = (int)(m / g.mcus_x);
    const int hv = g.hmax * g.vmax;
    if (b < hv) {
        *comp = 0;
        *bx = mcx * g.hmax + b % g.hmax;
        *by = mcy * g.vmax + b / g.hmax;
    } else {
        *comp = b - hv + 1;
        *bx = mcx;
        *by = mcy;
    }
    *mx = mcx;
}

// The block whose quantised DC the predictor of block `blk` holds: the previous block of the same component in the same restart
// interval, or -1 (the predictor is 0).
PN_JEHD long long dc_pred_block(const Geom &g, long long blk) {
    const long long m = blk / g.bpm;
    const int b = (int)(blk - m * g.bpm);
    const int hv = g.hmax * g.vmax;
    const int first = b < hv ? 0 : b, last = b < hv ? hv - 1 : b;
    if (b > first) return blk - 1;
    if (m == 0 || (g.rst > 0 && m % g.rst == 0)) return -1;
    return (m - 1) * g.bpm + last;
}

// An MCU padding block (compress_data's dummy blocks) is zero but for its DC, which is the quantised DC of the block before it in
// the MCU: at the right edge the last real block of its row, in a padding row at the bottom the last block of the row above it in
// the MCU (itself a copy when that is padding).  Returns false for a real block, else the real block (*sx, *sy) whose DC it takes.
PN_JEHD bool dummy_source(const Geom &g, int c, int bx, int by, int mx, int *sx, int *sy) {
    if (bx < g.bw[c] && by < g.bh[c]) return false;
    const int hc = c ? 1 : g.hmax;
    if (by >= g.bh[c]) {                                                // v <= 2: only the MCU's second row can be padding
        const int last = mx * hc + hc - 1;
        *sx = last < g.bw[c] - 1 ? last : g.bw[c] - 1;
        *sy = g.bh[c] - 1;
    } else {
        *sx = g.bw[c] - 1;
        *sy = by;
    }
    return true;
}

// ---- colour and sampling -------------------------------------------------------------------------------------------------------
// rgb_ycc_tab: FIX(x) = x * 2^16 + 0.5
PN_JEHD int ycc(int c, const uint8_t *bgr) {
    const int b = bgr[0], g = bgr[1], r = bgr[2];
    if (c == 0) return (19595 * r + 38470 * g + 7471 * b + 32768) >> 16;
    if (c == 1) return (-11059 * r - 21709 * g + 32768 * b + (128 << 16) + 32767) >> 16;
    return (32768 * r - 27439 * g - 5329 * b + (128 << 16) + 32767) >> 16;
}

// Component c's sample at (x, y) of its (downsampled, edge-expanded) plane; frame: BGR rows of w * 3 bytes.
// Horizontally the full-resolution rows are expanded before downsampling; vertically only to the downsampler's row group, the
// rows below the component's downsampled height repeating its last row.
PN_JEHD int sample(const Geom &g, const uint8_t *frame, int c, int x, int y) {
    const int hx = c ? g.hmax : 1, vy = c ? g.vmax : 1;
    const int dh = (g.h + vy - 1) / vy;
    if (y > dh - 1) y = dh - 1;
    int sum = 0;
    for (int v = 0; v < vy; ++v) {
        const int Y = y * vy + v < g.h - 1 ? y * vy + v : g.h - 1;
        for (int u = 0; u < hx; ++u) {
            const int X = x * hx + u < g.w - 1 ? x * hx + u : g.w - 1;
            sum += ycc(c, frame + ((long long)Y * g.w + X) * 3);
        }
    }
    if (hx == 1 && vy == 1) return sum;
    if (hx == 2 && vy == 1) return (sum + (x & 1)) >> 1;             // h2v1_downsample
    if (hx == 2 && vy == 2) return (sum + 1 + (x & 1)) >> 2;         // h2v2_downsample
    const int n = hx * vy;                                            // int_downsample
    return (sum + n / 2) / n;
}

// ---- forward DCT (jpeg_fdct_islow) -----------------------------------------------------------------------------------------------
#define PN_FIX_0_298631336 2446
#define PN_FIX_0_390180644 3196
#define PN_FIX_0_541196100 4433
#define PN_FIX_0_765366865 6270
#define PN_FIX_0_899976223 7373
#define PN_FIX_1_175875602 9633
#define PN_FIX_1_501321110 12299
#define PN_FIX_1_847759065 15137
#define PN_FIX_1_961570560 16069
#define PN_FIX_2_053119869 16819
#define PN_FIX_2_562915447 20995
#define PN_FIX_3_072711026 25172

PN_JEHD int descale(int x, int n) { return (x + (1 << (n - 1))) >> n; }

// One 8-point pass over d[0], d[s], .., d[7 s].  pass 0: rows (outputs scaled up by PASS1_BITS), 1: columns.
PN_JEHD void fdct_pass(int *d, int s, int pass) {
    const int CB = 13, P1 = 2;
    const int tmp0 = d[0] + d[7 * s], tmp7 = d[0] - d[7 * s];
    const int tmp1 = d[s] + d[6 * s], tmp6 = d[s] - d[6 * s];
    const int tmp2 = d[2 * s] + d[5 * s], tmp5 = d[2 * s] - d[5 * s];
    const int tmp3 = d[3 * s] + d[4 * s], tmp4 = d[3 * s] - d[4 * s];
    const int tmp10 = tmp0 + tmp3, tmp13 = tmp0 - tmp3, tmp11 = tmp1 + tmp2, tmp12 = tmp1 - tmp2;
    const int sh = pass == 0 ? CB - P1 : CB + P1;
    if (pass == 0) {
        d[0] = (tmp10 + tmp11) * (1 << P1);
        d[4 * s] = (tmp10 - tmp11) * (1 << P1);
    } else {
        d[0] = descale(tmp10 + tmp11, P1);
        d[4 * s] = descale(tmp10 - tmp11, P1);
    }
    int z1 = (tmp12 + tmp13) * PN_FIX_0_541196100;
    d[2 * s] = descale(z1 + tmp13 * PN_FIX_0_765366865, sh);
    d[6 * s] = descale(z1 + tmp12 * (-PN_FIX_1_847759065), sh);
    z1 = tmp4 + tmp7;
    int z2 = tmp5 + tmp6, z3 = tmp4 + tmp6, z4 = tmp5 + tmp7;
    const int z5 = (z3 + z4) * PN_FIX_1_175875602;
    const int t4 = tmp4 * PN_FIX_0_298631336, t5 = tmp5 * PN_FIX_2_053119869, t6 = tmp6 * PN_FIX_3_072711026,
              t7 = tmp7 * PN_FIX_1_501321110;
    z1 *= -PN_FIX_0_899976223;
    z2 *= -PN_FIX_2_562915447;
    z3 = z3 * -PN_FIX_1_961570560 + z5;
    z4 = z4 * -PN_FIX_0_390180644 + z5;
    d[7 * s] = descale(t4 + z1 + z3, sh);
    d[5 * s] = descale(t5 + z2 + z4, sh);
    d[3 * s] = descale(t6 + z2 + z3, sh);
    d[s] = descale(t7 + z1 + z4, sh);
}

// ---- quantisation ----------------------------------------------------------------------------------------------------------------
// compute_reciprocal (jcdctmgr.c) of a divisor d >= 2 with 16-bit DCTELEM: |x| -> ((|x| + corr) * recip) >> shift equals
// (|x| + d / 2) / d, the sign restored.
struct Recip {
    uint16_t recip, corr;
    uint8_t shift, pad;
};

PN_JEHD Recip compute_reciprocal(int d) {
    int b = 0;
    while ((2 << b) <= d) ++b;                                        // flss(d) - 1
    int r = 16 + b;
    uint32_t fq = (uint32_t)((1ull << r) / d);
    const uint32_t fr = (uint32_t)((1ull << r) % d);
    uint32_t c = d / 2;
    if (fr == 0) {
        fq >>= 1;
        --r;
    } else if (fr <= (uint32_t)d / 2u) {
        ++c;
    } else {
        ++fq;
    }
    Recip q;
    q.recip = (uint16_t)fq;
    q.corr = (uint16_t)c;
    q.shift = (uint8_t)r;
    q.pad = 0;
    return q;
}

PN_JEHD int quantize(int x, Recip q) {
    const uint32_t a = (uint32_t)(x < 0 ? -x : x);
    const int t = (int)(((uint32_t)(uint16_t)(a + q.corr) * q.recip) >> q.shift);
    return x < 0 ? -t : t;
}

// ---- tables ------------------------------------------------------------------------------------------------------------------------
// natural index -> zig-zag index is the inverse of jpeg_natural_order
#define PN_JPEG_ZIGZAG_OF_NATURAL {                                                                                      \
    0, 1, 5, 6, 14, 15, 27, 28, 2, 4, 7, 13, 16, 26, 29, 42, 3, 8, 12, 17, 25, 30, 41, 43, 9, 11, 18, 24, 31, 40, 44, 53,  \
    10, 19, 23, 32, 39, 45, 52, 54, 20, 22, 33, 38, 46, 51, 55, 60, 21, 34, 37, 47, 50, 56, 59, 61, 35, 36, 48, 49, 57, 58, \
    62, 63 }
#ifdef __CUDACC__
__device__ const uint8_t kZigzagDev[64] = PN_JPEG_ZIGZAG_OF_NATURAL;
#endif
static const uint8_t kZigzagHost[64] = PN_JPEG_ZIGZAG_OF_NATURAL;

PN_JEHD int zigzag_of(int natural) {
#ifdef __CUDA_ARCH__
    return kZigzagDev[natural];
#else
    return kZigzagHost[natural];
#endif
}

// Encoder-side tables of one call, passed by value to the kernels (so a captured graph keeps them).
struct HuffEnc {
    uint16_t code[256];
    uint8_t size[256];     // 0: symbol not in the table
};
struct Tables {
    Recip quant[2][64];    // luma, chroma; natural order
    uint16_t qval[2][64];  // qtbl entries, natural order
    HuffEnc dc[2], ac[2];
};

// ---- entropy coding (encode_one_block) --------------------------------------------------------------------------------------------
PN_JEHD int nbits(int a) {                                          // a >= 0: JPEG_NBITS
    int n = 0;
    while (a) {
        ++n;
        a >>= 1;
    }
    return n;
}

// Emit one block (coefficients in zig-zag order) with DC difference `diff` into `put(code, size)`.
template <typename Put>
PN_JEHD void encode_block(const int16_t *zz, int diff, const HuffEnc &dc, const HuffEnc &ac, Put &put) {
    {
        const int a = diff < 0 ? -diff : diff, n = nbits(a);
        put((uint32_t)dc.code[n], dc.size[n]);
        if (n) put((uint32_t)(diff < 0 ? diff - 1 : diff) & ((1u << n) - 1u), n);
    }
    int r = 0;
    for (int k = 1; k < 64; ++k) {
        const int v = zz[k];
        if (v == 0) {
            ++r;
            continue;
        }
        while (r > 15) {
            put((uint32_t)ac.code[0xF0], ac.size[0xF0]);
            r -= 16;
        }
        const int a = v < 0 ? -v : v, n = nbits(a);
        const int sym = (r << 4) + n;
        put((uint32_t)ac.code[sym], ac.size[sym]);
        put((uint32_t)(v < 0 ? v - 1 : v) & ((1u << n) - 1u), n);
        r = 0;
    }
    if (r > 0) put((uint32_t)ac.code[0], ac.size[0]);
}

struct CountBits {
    uint32_t bits = 0;
    PN_JEHD void operator()(uint32_t, int n) { bits += (uint32_t)n; }
};

// Worst case of one block: DC 16 + 11 bits, 63 AC symbols of 16 + 10 bits.
constexpr int kMaxBlockBits = 16 + 11 + 63 * (16 + 10);

}  // namespace jpege
}  // namespace pn

// ---- host only: tables and headers ----------------------------------------------------------------------------------------------------
#include <string.h>
namespace pn {
namespace jpege {

static const uint8_t kStdQuant[2][64] = {   // jcparam.c std_luminance_quant_tbl / std_chrominance_quant_tbl, natural order
    {16, 11, 10, 16, 24, 40, 51, 61, 12, 12, 14, 19, 26, 58, 60, 55, 14, 13, 16, 24, 40, 57, 69, 56, 14, 17, 22, 29, 51, 87, 80, 62,
     18, 22, 37, 56, 68, 109, 103, 77, 24, 35, 55, 64, 81, 104, 113, 92, 49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100,
     103, 99},
    {17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99, 24, 26, 56, 99, 99, 99, 99, 99, 47, 66, 99, 99, 99, 99, 99, 99,
     99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99}};

// jstdhuff.c: bits[1..16] and values of DC luma, AC luma, DC chroma, AC chroma
static const uint8_t kStdBits[4][17] = {
    {0, 0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0},
    {0, 0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7d},
    {0, 0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0},
    {0, 0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 0x77}};
static const uint8_t kStdDcVals[12] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11};
static const uint8_t kStdAcLuma[162] = {
    0x01, 0x02, 0x03, 0x00, 0x04, 0x11, 0x05, 0x12, 0x21, 0x31, 0x41, 0x06, 0x13, 0x51, 0x61, 0x07, 0x22, 0x71, 0x14, 0x32, 0x81,
    0x91, 0xa1, 0x08, 0x23, 0x42, 0xb1, 0xc1, 0x15, 0x52, 0xd1, 0xf0, 0x24, 0x33, 0x62, 0x72, 0x82, 0x09, 0x0a, 0x16, 0x17, 0x18,
    0x19, 0x1a, 0x25, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x34, 0x35, 0x36, 0x37, 0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48,
    0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59, 0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75,
    0x76, 0x77, 0x78, 0x79, 0x7a, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99,
    0x9a, 0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3,
    0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe1, 0xe2, 0xe3, 0xe4, 0xe5,
    0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf1, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa};
static const uint8_t kStdAcChroma[162] = {
    0x00, 0x01, 0x02, 0x03, 0x11, 0x04, 0x05, 0x21, 0x31, 0x06, 0x12, 0x41, 0x51, 0x07, 0x61, 0x71, 0x13, 0x22, 0x32, 0x81, 0x08,
    0x14, 0x42, 0x91, 0xa1, 0xb1, 0xc1, 0x09, 0x23, 0x33, 0x52, 0xf0, 0x15, 0x62, 0x72, 0xd1, 0x0a, 0x16, 0x24, 0x34, 0xe1, 0x25,
    0xf1, 0x17, 0x18, 0x19, 0x1a, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x35, 0x36, 0x37, 0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47,
    0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59, 0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74,
    0x75, 0x76, 0x77, 0x78, 0x79, 0x7a, 0x82, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97,
    0x98, 0x99, 0x9a, 0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba,
    0xc2, 0xc3, 0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe2, 0xe3, 0xe4,
    0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa};

inline const uint8_t *std_vals(int t) { return t == 1 ? kStdAcLuma : t == 3 ? kStdAcChroma : kStdDcVals; }

// jpeg_quality_scaling + jpeg_add_quant_table (force_baseline): cv2 clamps its quality to 0..100 first
inline void quant_table(int quality, int which, uint16_t *q) {
    if (quality <= 0) quality = 1;
    if (quality > 100) quality = 100;
    const int scale = quality < 50 ? 5000 / quality : 200 - quality * 2;
    for (int k = 0; k < 64; ++k) {
        long t = ((long)kStdQuant[which][k] * scale + 50L) / 100L;
        q[k] = (uint16_t)(t < 1 ? 1 : t > 255 ? 255 : t);
    }
}

// jpeg_make_c_derived_tbl: canonical codes from bits / values
inline void derive_huff(int t, HuffEnc *h) {
    memset(h, 0, sizeof(*h));
    const uint8_t *vals = std_vals(t);
    uint32_t code = 0;
    int p = 0;
    for (int l = 1; l <= 16; ++l) {
        for (int i = 0; i < kStdBits[t][l]; ++i, ++p) {
            h->code[vals[p]] = (uint16_t)code++;
            h->size[vals[p]] = (uint8_t)l;
        }
        code <<= 1;
    }
}

inline void make_tables(int quality, Tables *T) {
    for (int w = 0; w < 2; ++w) {
        quant_table(quality, w, T->qval[w]);
        for (int k = 0; k < 64; ++k) T->quant[w][k] = compute_reciprocal(8 * T->qval[w][k]);
    }
    derive_huff(0, &T->dc[0]);
    derive_huff(1, &T->ac[0]);
    derive_huff(2, &T->dc[1]);
    derive_huff(3, &T->ac[1]);
}

constexpr int kMaxHeader = 1024;

// Everything before the entropy-coded data, as jcmarker.c writes it for cv2.  Returns the length; *sof_hw is the offset of the
// SOF0 height (big-endian; the width follows), patched per image.
inline int write_header(const Tables &T, int sampling, int rst, int h, int w, uint8_t *o, int *sof_hw) {
    int n = 0, hm = 1, vm = 1;
    luma_factors(sampling, &hm, &vm);
    auto b = [&](int v) { o[n++] = (uint8_t)v; };
    auto w16 = [&](int v) { b(v >> 8); b(v & 0xFF); };
    w16(0xFFD8);
    w16(0xFFE0); w16(16);
    b('J'); b('F'); b('I'); b('F'); b(0);
    b(1); b(1); b(0); w16(1); w16(1); b(0); b(0);
    for (int t = 0; t < 2; ++t) {
        w16(0xFFDB); w16(67); b(t);
        for (int z = 0; z < 64; ++z) {
            int nat = 0;
            while (zigzag_of(nat) != z) ++nat;
            b(T.qval[t][nat]);
        }
    }
    w16(0xFFC0); w16(17); b(8);
    *sof_hw = n;
    w16(h); w16(w);
    b(3);
    b(1); b((hm << 4) | vm); b(0);
    b(2); b(0x11); b(1);
    b(3); b(0x11); b(1);
    for (int t = 0; t < 4; ++t) {
        int nv = 0;
        for (int l = 1; l <= 16; ++l) nv += kStdBits[t][l];
        w16(0xFFC4); w16(2 + 1 + 16 + nv);
        b((t & 1) << 4 | (t >> 1));
        for (int l = 1; l <= 16; ++l) b(kStdBits[t][l]);
        for (int i = 0; i < nv; ++i) b(std_vals(t)[i]);
    }
    if (rst > 0) {
        w16(0xFFDD); w16(4); w16(rst);
    }
    w16(0xFFDA); w16(12); b(3);
    b(1); b(0x00);
    b(2); b(0x11);
    b(3); b(0x11);
    b(0); b(63); b(0);
    return n;
}

// A true worst case of one file: header, every restart interval at kMaxBlockBits per block padded to a byte and every byte
// stuffed, the RST markers and EOI.
inline long long encode_bound(const Geom &g, int header_bytes) {
    if (g.nblk == 0) return 0;
    const long long mcus = (long long)g.mcus_x * g.mcus_y;
    const long long per = g.rst > 0 ? g.rst : mcus;
    long long total = header_bytes + 2;
    for (long long m0 = 0; m0 < mcus; m0 += per) {
        const long long m = mcus - m0 < per ? mcus - m0 : per;
        total += 2 * ((m * g.bpm * kMaxBlockBits + 7) / 8) + 2;
    }
    return total;
}

}  // namespace jpege
}  // namespace pn
