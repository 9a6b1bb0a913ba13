// Baseline JPEG decode arithmetic, restated from libjpeg-turbo 3.1 (what cv2 4.13 runs for cv2.imread / cv2.imdecode with
// IMREAD_COLOR), as __host__ __device__ functions: csrc/jpeg.cu runs them in parallel, tests/test_jpeg_cpu.py compiles them
// into a serial host decoder and compares it with cv2 byte for byte.
//
//   entropy data:  byte de-stuffing and markers (jdhuff.c fill_bit_buffer), Huffman symbols (HUFF_DECODE / jpeg_huff_decode),
//                  HUFF_EXTEND, zig-zag runs landing on coefficient 63 past the end (jpeg_natural_order's 16 extra entries)
//   IDCT:          jpeg_idct_islow (jidctint.c): CONST_BITS 13, PASS1_BITS 2, range_limit[x & RANGE_MASK]; at 1/2, 1/4, 1/8
//                  (cv2's IMREAD_REDUCED_COLOR_*) jpeg_idct_4x4 / 2x2 / 1x1 (jidctred.c) with the per-component scaled sizes
//                  of jdmaster.c
//   upsampling:    jdsample.c h2v1 / h1v2 / h2v2 fancy, replication otherwise, chosen from the scaled group ratios; context
//                  rows as jdmainct.c supplies them
//   colour:        jdcolor.c ycc_rgb_convert (build_ycc_rgb_table, SCALEBITS 16) into B, G, R; grayscale replicated
//   orientation:   the EXIF flips / transposes cv2.imread applies to the decoded frame, as a map of output to source pixels
#pragma once
#include <stdint.h>

#include "../../include/posenet_b200.h"

#ifdef __CUDACC__
#define PN_JHD __host__ __device__ __forceinline__
#else
#define PN_JHD inline
#endif

namespace pn {
namespace jpeg {

// jpeg_natural_order (jutils.c): zig-zag index -> natural index, with 16 extra entries of 63 for corrupt runs
#define PN_JPEG_NATURAL_ORDER {                                                                                         \
    0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21, 28, \
    35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47,  \
    55, 62, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63 }
#ifdef __CUDACC__
__device__ const uint8_t kNaturalDev[80] = PN_JPEG_NATURAL_ORDER;
#endif
static const uint8_t kNaturalHost[80] = PN_JPEG_NATURAL_ORDER;

PN_JHD int natural_order(int k) {
#ifdef __CUDA_ARCH__
    return kNaturalDev[k];
#else
    return kNaturalHost[k];
#endif
}

// ---- entropy-coded segment: de-stuffing ------------------------------------------------------------------------------------
// A byte of the scan is classified from itself and its neighbours alone, so every byte can be classified in parallel:
// 0xFF 0x00 is a data 0xFF (a run of 0xFF fill bytes before the 0x00 collapses into it, as fill_bit_buffer reads it), 0xFF
// followed by 0xD0..0xD7 a restart marker, 0xFF followed by anything else but 0xFF the end of the scan.
enum { BYTE_DATA = 0, BYTE_DROP = 1, BYTE_RST = 2, BYTE_END = 3 };
// prev / next: -1 when outside the scan (before its first byte, past the end of the file)
PN_JHD int classify_byte(int prev, int b, int next) {
    if (b == 0xFF) {
        if (next == 0x00) return BYTE_DATA;
        if (next == 0xFF) return BYTE_DROP;
        if (next >= 0xD0 && next <= 0xD7) return BYTE_RST;
        return BYTE_END;                       // a marker, or the file ends on 0xFF
    }
    return prev == 0xFF ? BYTE_DROP : BYTE_DATA;
}

// ---- Huffman decode ----------------------------------------------------------------------------------------------------------
// Bits of a de-stuffed segment, MSB first; bits past `nbytes` read as zero (what libjpeg inserts after a marker).
struct BitSrc {
    const uint8_t *p;
    uint32_t nbytes;
    PN_JHD uint32_t peek32(uint32_t pos) const {
        const uint32_t q = pos >> 3;
        uint64_t w = 0;
#pragma unroll
        for (int i = 0; i < 5; ++i) w = (w << 8) | (q + i < nbytes ? p[q + i] : 0u);
        return (uint32_t)(w >> (8 - (pos & 7)));
    }
};

// One symbol at the top of `bits` (the 32 bits at the current position).  Returns the code length, 0 for a code not in the table
// (jpeg_huff_decode's JWRN_HUFF_BAD_CODE).
PN_JHD int huff_symbol(const pn_jpeg_huff &t, uint32_t bits, int *sym) {
    const int e = t.lookup[bits >> 24];
    if (e) {
        *sym = e & 0xFF;
        return e >> 8;
    }
    int l = 9;
    int32_t code = (int32_t)(bits >> 23);
    while (l <= 16 && code > t.maxcode[l]) {
        ++l;
        code = (int32_t)(bits >> (32 - l));
    }
    if (l > 16) return 0;
    *sym = t.huffval[(code + t.valoffset[l]) & 0xFF];
    return l;
}

PN_JHD int huff_extend(uint32_t r, int s) {    // HUFF_EXTEND(x, s), s in 1..15
    return (int)r < (1 << (s - 1)) ? (int)r + (int)((~0u << s) + 1u) : (int)r;
}

// Decoder position at a codeword boundary: bit offset in the segment, block within the MCU, zig-zag index (0: next is a DC).
struct State {
    uint32_t pos;
    int b, z;
};
PN_JHD uint64_t pack(const State &s) { return ((uint64_t)s.pos << 16) | ((uint64_t)s.b << 8) | (uint64_t)s.z; }
PN_JHD State unpack(uint64_t v) { return State{(uint32_t)(v >> 16), (int)((v >> 8) & 0xFF), (int)(v & 0xFF)}; }
constexpr uint64_t kBadState = ~0ull;   // a path that met a code not in its table

// One codeword (and its extra bits).  Returns false on a bad code.  *started is set when the codeword begins a block.
PN_JHD bool step(const pn_jpeg_desc &d, const BitSrc &src, State &s, bool *started) {
    const pn_jpeg_comp &c = d.comp[d.mcu_comp[s.b]];
    const uint32_t bits = src.peek32(s.pos);
    int sym;
    if (s.z == 0) {
        const int len = huff_symbol(d.huff[c.dc], bits, &sym);
        if (!len) return false;
        s.pos += len + sym;
        s.z = 1;
        *started = true;
        return true;
    }
    *started = false;
    const int len = huff_symbol(d.huff[c.ac], bits, &sym);
    if (!len) return false;
    const int r = sym >> 4, sz = sym & 15;
    s.pos += len;
    if (sz) {
        s.pos += sz;
        s.z += r + 1;
    } else if (r == 15) {
        s.z += 16;
    } else {
        s.z = 64;                               // EOB
    }
    if (s.z >= 64) {
        s.z = 0;
        s.b = s.b + 1 == d.blocks_per_mcu ? 0 : s.b + 1;
    }
    return true;
}

// Decode from `s` until the first codeword boundary at or past `end`; *blocks += blocks begun on the way.  False on a bad code.
PN_JHD bool advance(const pn_jpeg_desc &d, const BitSrc &src, State &s, uint32_t end, uint32_t *blocks) {
    while (s.pos < end) {
        bool started;
        if (!step(d, src, s, &started)) return false;
        *blocks += started;
    }
    return true;
}

// Self-synchronisation across subsequences of `sub_bits` bits (0 .. nk-1; boundaries at the ends of 0 .. nk-2).  `s` is a path's
// state at the end of subsequence k.  The path is followed through the next subsequences until its state at the end of some
// subsequence j equals e1(j), the exit of j's speculative decode: from there on the two paths are one.  Returns j, MERGE_TAIL
// when no boundary is left (the path owns the rest of the segment), MERGE_NONE after `limit` subsequences or a bad code.
// *blocks: blocks begun between the end of k and the end of j.
constexpr int MERGE_NONE = -1, MERGE_TAIL = -2;
template <class E1>
PN_JHD int merge_point(const pn_jpeg_desc &d, const BitSrc &src, State s, int k, int nk, uint32_t sub_bits, int limit, E1 e1,
                       uint32_t *blocks) {
    *blocks = 0;
    for (int j = k + 1; j < nk - 1; ++j) {
        if (j - k > limit || !advance(d, src, s, (uint32_t)(j + 1) * sub_bits, blocks)) return MERGE_NONE;
        if (pack(s) == e1(j)) return j;
    }
    return MERGE_TAIL;
}

// Finish the block `s` is inside (z != 0) without storing it.
PN_JHD bool skip_rest_of_block(const pn_jpeg_desc &d, const BitSrc &src, State &s) {
    while (s.z != 0) {
        bool started;
        if (!step(d, src, s, &started)) return false;
    }
    return true;
}

// One whole block from its DC codeword (s.z == 0), stored as jdhuff.c's decode_mcu stores it into a zeroed JBLOCK: blk[0] is the
// DC DIFFERENCE (the per-component running sum is added afterwards), AC values at natural positions.  `blk` has 64 JCOEFs.
PN_JHD bool decode_block(const pn_jpeg_desc &d, const BitSrc &src, State &s, int16_t *blk) {
    const pn_jpeg_comp &c = d.comp[d.mcu_comp[s.b]];
#ifdef __CUDA_ARCH__
#pragma unroll
    for (int k = 0; k < 8; ++k) reinterpret_cast<uint4 *>(blk)[k] = make_uint4(0, 0, 0, 0);   // blk is 128-byte aligned
#else
    for (int k = 0; k < 64; ++k) blk[k] = 0;
#endif
    uint32_t bits = src.peek32(s.pos);
    int sym;
    int len = huff_symbol(d.huff[c.dc], bits, &sym);
    if (!len) return false;
    s.pos += len;
    int v = 0;
    if (sym) {
        v = huff_extend(src.peek32(s.pos) >> (32 - sym), sym);
        s.pos += sym;
    }
    blk[0] = (int16_t)v;
    const pn_jpeg_huff &ac = d.huff[c.ac];
    for (int k = 1; k < 64; ++k) {
        bits = src.peek32(s.pos);
        len = huff_symbol(ac, bits, &sym);
        if (!len) return false;
        s.pos += len;
        const int r = sym >> 4, sz = sym & 15;
        if (sz) {
            k += r;
            blk[natural_order(k)] = (int16_t)huff_extend((bits << len) >> (32 - sz), sz);
            s.pos += sz;
        } else {
            if (r != 15) break;
            k += 15;
        }
    }
    s.z = 0;
    s.b = s.b + 1 == d.blocks_per_mcu ? 0 : s.b + 1;
    return true;
}

// ---- IDCT: jpeg_idct_islow -------------------------------------------------------------------------------------------------------
constexpr int CONST_BITS = 13, PASS1_BITS = 2;
constexpr int64_t FIX_0_298631336 = 2446, FIX_0_390180644 = 3196, FIX_0_541196100 = 4433, FIX_0_765366865 = 6270,
                  FIX_0_899976223 = 7373, FIX_1_175875602 = 9633, FIX_1_501321110 = 12299, FIX_1_847759065 = 15137,
                  FIX_1_961570560 = 16069, FIX_2_053119869 = 16819, FIX_2_562915447 = 20995, FIX_3_072711026 = 25172;

PN_JHD int64_t descale(int64_t x, int n) { return (x + ((int64_t)1 << (n - 1))) >> n; }

// range_limit[x & RANGE_MASK] of the post-IDCT table prepare_range_limit_table builds (x centred on 0)
PN_JHD uint8_t idct_limit(int64_t x) {
    const int i = (int)(x & 1023);
    return (uint8_t)(i < 128 ? i + 128 : i < 512 ? 255 : i < 896 ? 0 : i - 896);
}

// The 1-D butterfly both passes share: in[0..7] (already dequantised / from the work array) -> the eight sums before descaling.
PN_JHD void idct_1d(const int64_t in[8], int64_t out[8]) {
    int64_t z2 = in[2], z3 = in[6];
    int64_t z1 = (z2 + z3) * FIX_0_541196100;
    int64_t tmp2 = z1 + z3 * -FIX_1_847759065;
    int64_t tmp3 = z1 + z2 * FIX_0_765366865;
    int64_t tmp0 = (in[0] + in[4]) * ((int64_t)1 << CONST_BITS);
    int64_t tmp1 = (in[0] - in[4]) * ((int64_t)1 << CONST_BITS);
    const int64_t tmp10 = tmp0 + tmp3, tmp13 = tmp0 - tmp3, tmp11 = tmp1 + tmp2, tmp12 = tmp1 - tmp2;
    tmp0 = in[7]; tmp1 = in[5]; tmp2 = in[3]; tmp3 = in[1];
    z1 = tmp0 + tmp3;
    z2 = tmp1 + tmp2;
    z3 = tmp0 + tmp2;
    int64_t z4 = tmp1 + tmp3;
    const int64_t z5 = (z3 + z4) * FIX_1_175875602;
    tmp0 *= FIX_0_298631336;
    tmp1 *= FIX_2_053119869;
    tmp2 *= FIX_3_072711026;
    tmp3 *= FIX_1_501321110;
    z1 *= -FIX_0_899976223;
    z2 *= -FIX_2_562915447;
    z3 *= -FIX_1_961570560;
    z4 *= -FIX_0_390180644;
    z3 += z5;
    z4 += z5;
    tmp0 += z1 + z3;
    tmp1 += z2 + z4;
    tmp2 += z2 + z3;
    tmp3 += z1 + z4;
    out[0] = tmp10 + tmp3; out[7] = tmp10 - tmp3;
    out[1] = tmp11 + tmp2; out[6] = tmp11 - tmp2;
    out[2] = tmp12 + tmp1; out[5] = tmp12 - tmp1;
    out[3] = tmp13 + tmp0; out[4] = tmp13 - tmp0;
}

// Pass 1 for column `col`: coef (natural order JCOEFs) x quant -> ws[row * 8 + col] (int, as libjpeg's workspace)
PN_JHD void idct_column(const int16_t *coef, const int16_t *quant, int col, int *ws) {
    int64_t in[8], out[8];
    bool ac_zero = true;
    for (int r = 0; r < 8; ++r) {
        in[r] = (int64_t)((int)coef[r * 8 + col] * (int)quant[r * 8 + col]);
        if (r && coef[r * 8 + col]) ac_zero = false;
    }
    if (ac_zero) {                              // the AC-free column shortcut (exactly what the full pass computes)
        for (int r = 0; r < 8; ++r) ws[r * 8 + col] = (int)(in[0] * (1 << PASS1_BITS));
        return;
    }
    idct_1d(in, out);
    for (int r = 0; r < 8; ++r) ws[r * 8 + col] = (int)descale(out[r], CONST_BITS - PASS1_BITS);
}

// Pass 2 for row `row` of the work array -> 8 samples
PN_JHD void idct_row(const int *ws, int row, uint8_t *outp) {
    int64_t in[8], out[8];
    for (int c = 0; c < 8; ++c) in[c] = ws[row * 8 + c];
    idct_1d(in, out);
    for (int c = 0; c < 8; ++c) outp[c] = idct_limit(descale(out[c], CONST_BITS + PASS1_BITS + 3));
}

// ---- reduced IDCTs: jidctred.c (cv2's IMREAD_REDUCED_*: libjpeg's DCT-domain scaling) ------------------------------------------
// jpeg_idct_4x4 and jpeg_idct_2x2 are their own transforms, not truncations of islow: they read the odd coefficients 1, 3, 5, 7
// (and 2, 6 for 4x4) and never coefficient 4.  Both passes split like idct_column / idct_row: pass 1 fills ws[r * 8 + col] for
// r < n (columns the second pass does not read are skipped), pass 2 turns row `row` of ws into n samples.
constexpr int64_t FIX_0_211164243 = 1730, FIX_0_509795579 = 4176, FIX_0_601344887 = 4926, FIX_0_720959822 = 5906,
                  FIX_0_850430095 = 6967, FIX_1_061594337 = 8697, FIX_1_272758580 = 10426, FIX_1_451774981 = 11893,
                  FIX_2_172734803 = 17799, FIX_3_624509785 = 29692;

// The 4-point odd part both passes of jpeg_idct_4x4 share (z1..z4: inputs 7, 5, 3, 1).
PN_JHD void idct4_odd(int64_t z1, int64_t z2, int64_t z3, int64_t z4, int64_t *tmp0, int64_t *tmp2) {
    *tmp0 = z1 * -FIX_0_211164243 + z2 * FIX_1_451774981 + z3 * -FIX_2_172734803 + z4 * FIX_1_061594337;
    *tmp2 = z1 * -FIX_0_509795579 + z2 * -FIX_0_601344887 + z3 * FIX_0_899976223 + z4 * FIX_2_562915447;
}

PN_JHD void idct4x4_column(const int16_t *coef, const int16_t *quant, int col, int *ws) {
    if (col == 4) return;
    auto dq = [&](int r) { return (int64_t)((int)coef[r * 8 + col] * (int)quant[r * 8 + col]); };
    const int64_t tmp0e = dq(0) * ((int64_t)1 << (CONST_BITS + 1));
    const int64_t tmp2e = dq(2) * FIX_1_847759065 + dq(6) * -FIX_0_765366865;
    const int64_t tmp10 = tmp0e + tmp2e, tmp12 = tmp0e - tmp2e;
    int64_t tmp0, tmp2;
    idct4_odd(dq(7), dq(5), dq(3), dq(1), &tmp0, &tmp2);
    const int sh = CONST_BITS - PASS1_BITS + 1;   // the all-AC-zero shortcut of jidctred.c computes the same values
    ws[0 * 8 + col] = (int)descale(tmp10 + tmp2, sh);
    ws[3 * 8 + col] = (int)descale(tmp10 - tmp2, sh);
    ws[1 * 8 + col] = (int)descale(tmp12 + tmp0, sh);
    ws[2 * 8 + col] = (int)descale(tmp12 - tmp0, sh);
}

PN_JHD void idct4x4_row(const int *ws, int row, uint8_t *outp) {
    const int *w = ws + row * 8;
    const int64_t tmp0e = (int64_t)w[0] * ((int64_t)1 << (CONST_BITS + 1));
    const int64_t tmp2e = (int64_t)w[2] * FIX_1_847759065 + (int64_t)w[6] * -FIX_0_765366865;
    const int64_t tmp10 = tmp0e + tmp2e, tmp12 = tmp0e - tmp2e;
    int64_t tmp0, tmp2;
    idct4_odd(w[7], w[5], w[3], w[1], &tmp0, &tmp2);
    const int sh = CONST_BITS + PASS1_BITS + 3 + 1;
    outp[0] = idct_limit(descale(tmp10 + tmp2, sh));
    outp[3] = idct_limit(descale(tmp10 - tmp2, sh));
    outp[1] = idct_limit(descale(tmp12 + tmp0, sh));
    outp[2] = idct_limit(descale(tmp12 - tmp0, sh));
}

PN_JHD void idct2x2_column(const int16_t *coef, const int16_t *quant, int col, int *ws) {
    if (col == 2 || col == 4 || col == 6) return;
    auto dq = [&](int r) { return (int64_t)((int)coef[r * 8 + col] * (int)quant[r * 8 + col]); };
    const int64_t tmp10 = dq(0) * ((int64_t)1 << (CONST_BITS + 2));
    const int64_t tmp0 = dq(7) * -FIX_0_720959822 + dq(5) * FIX_0_850430095 + dq(3) * -FIX_1_272758580 + dq(1) * FIX_3_624509785;
    ws[0 * 8 + col] = (int)descale(tmp10 + tmp0, CONST_BITS - PASS1_BITS + 2);
    ws[1 * 8 + col] = (int)descale(tmp10 - tmp0, CONST_BITS - PASS1_BITS + 2);
}

PN_JHD void idct2x2_row(const int *ws, int row, uint8_t *outp) {
    const int *w = ws + row * 8;
    const int64_t tmp10 = (int64_t)w[0] * ((int64_t)1 << (CONST_BITS + 2));
    const int64_t tmp0 = (int64_t)w[7] * -FIX_0_720959822 + (int64_t)w[5] * FIX_0_850430095 +
                         (int64_t)w[3] * -FIX_1_272758580 + (int64_t)w[1] * FIX_3_624509785;
    outp[0] = idct_limit(descale(tmp10 + tmp0, CONST_BITS + PASS1_BITS + 3 + 2));
    outp[1] = idct_limit(descale(tmp10 - tmp0, CONST_BITS + PASS1_BITS + 3 + 2));
}

// jpeg_idct_1x1: the DC term alone, descaled by 3
PN_JHD uint8_t idct1x1(const int16_t *coef, const int16_t *quant) {
    return idct_limit(descale((int64_t)((int)coef[0] * (int)quant[0]), 3));
}

// The IDCT of scaled size n (8: islow, 4, 2, 1), split in passes as above; idct_row_scaled writes n samples.
PN_JHD void idct_column_scaled(const int16_t *coef, const int16_t *quant, int n, int col, int *ws) {
    if (n == 8) idct_column(coef, quant, col, ws);
    else if (n == 4) idct4x4_column(coef, quant, col, ws);
    else if (n == 2) idct2x2_column(coef, quant, col, ws);
}
PN_JHD void idct_row_scaled(const int16_t *coef, const int16_t *quant, const int *ws, int n, int row, uint8_t *outp) {
    if (n == 8) idct_row(ws, row, outp);
    else if (n == 4) idct4x4_row(ws, row, outp);
    else if (n == 2) idct2x2_row(ws, row, outp);
    else outp[0] = idct1x1(coef, quant);
}

// ---- output geometry at 1 / scale_denom (jdmaster.c jpeg_core_output_dimensions, jdsample.c jinit_upsampler) ----------------------
// The frame is ceil(h / d) x ceil(w / d).  Luma's IDCT is 8 / d; a component whose samples are coarser than the largest factor
// doubles its IDCT size while that keeps the ratio to the minimum integral in both directions, so (e.g.) 4:2:0 chroma at 1/2 is
// decoded with the full 8x8 IDCT and needs no upsampling.  What is left to upsample is the ratio of max_h x max_v output samples
// to the component's h_in_group x v_in_group; fancy filters only when the minimum scaled size is above 1.
enum { UP_FULL = 0, UP_H2V1_FANCY, UP_H1V2_FANCY, UP_H2V2_FANCY, UP_REPLICATE };
struct CompScale {
    int ssize;        // DCT_scaled_size: samples per block side
    int hr, vr;       // upsampling ratios (output samples per component sample)
    int dw, dh;       // downsampled_width / downsampled_height: the component's real samples at this scale
    int up;           // UP_*
};
struct Scaled {
    int h, w;         // output frame size
    CompScale comp[3];
};

PN_JHD bool valid_denom(int denom) { return denom == 1 || denom == 2 || denom == 4 || denom == 8; }

// DCT_scaled_size of component c (sampling factors >= 1, denom valid)
PN_JHD int comp_ssize(const pn_jpeg_desc &d, int denom, int c) {
    const int mn = 8 / denom;
    if (mn == 8) return 8;
    int max_h = 1, max_v = 1;
    for (int k = 0; k < d.ncomp; ++k) {
        max_h = d.comp[k].h > max_h ? d.comp[k].h : max_h;
        max_v = d.comp[k].v > max_v ? d.comp[k].v : max_v;
    }
    const int h = d.comp[c].h, v = d.comp[c].v;
    int ss = mn;
    while (ss < 8 && (max_h * mn) % (h * ss * 2) == 0 && (max_v * mn) % (v * ss * 2) == 0) ss *= 2;
    return ss;
}

// False for a scale_denom other than 1, 2, 4, 8 or a ratio that is not integral (JERR_FRACT_SAMPLE_NOTIMPL).
PN_JHD bool scaled_geometry(const pn_jpeg_desc &d, int denom, Scaled *g) {
    if (!valid_denom(denom)) return false;
    const int mn = 8 / denom;
    int max_h = 1, max_v = 1;
    for (int c = 0; c < d.ncomp; ++c) {
        if (d.comp[c].h < 1 || d.comp[c].v < 1) return false;
        max_h = d.comp[c].h > max_h ? d.comp[c].h : max_h;
        max_v = d.comp[c].v > max_v ? d.comp[c].v : max_v;
    }
    g->h = (d.height + denom - 1) / denom;
    g->w = (d.width + denom - 1) / denom;
    for (int c = 0; c < 3; ++c) {
        CompScale &s = g->comp[c];
        s = CompScale{mn, 1, 1, 1, 1, UP_FULL};
        if (c >= d.ncomp) continue;
        const int h = d.comp[c].h, v = d.comp[c].v;
        const int ss = comp_ssize(d, denom, c);
        s.ssize = ss;
        s.dw = (int)(((int64_t)d.width * h * ss + max_h * 8 - 1) / (max_h * 8));
        s.dh = (int)(((int64_t)d.height * v * ss + max_v * 8 - 1) / (max_v * 8));
        const int hin = h * ss / mn, vin = v * ss / mn;
        if (max_h % hin || max_v % vin) return false;
        s.hr = max_h / hin;
        s.vr = max_v / vin;
        const bool fancy = mn > 1;
        if (s.hr == 1 && s.vr == 1) s.up = UP_FULL;
        else if (s.hr == 2 && s.vr == 1) s.up = fancy && s.dw > 2 ? UP_H2V1_FANCY : UP_REPLICATE;
        else if (s.hr == 1 && s.vr == 2) s.up = fancy ? UP_H1V2_FANCY : UP_REPLICATE;
        else if (s.hr == 2 && s.vr == 2) s.up = fancy && s.dw > 2 ? UP_H2V2_FANCY : UP_REPLICATE;
        else s.up = UP_REPLICATE;
    }
    return true;
}

// ---- upsampling (jdsample.c) -------------------------------------------------------------------------------------------------------
// Sample (y, x) of the output-resolution component, from its downsampled plane (pitch bytes per row, dw x dh real samples).
// Rows above the first and below row dh - 1 are that row repeated (jdmainct.c context rows).
PN_JHD int upsample(const uint8_t *pl, int pitch, const CompScale &c, int y, int x) {
    const int dw = c.dw, dh = c.dh;
    switch (c.up) {
    case UP_FULL: return pl[(int64_t)y * pitch + x];
    case UP_H1V2_FANCY: {                                                            // h1v2_fancy_upsample
        const int iy = y >> 1, v = y & 1;
        const int nb = v ? (iy + 1 < dh ? iy + 1 : dh - 1) : (iy > 0 ? iy - 1 : 0);
        return (3 * pl[(int64_t)iy * pitch + x] + pl[(int64_t)nb * pitch + x] + (v ? 2 : 1)) >> 2;
    }
    case UP_H2V1_FANCY: {                                                            // h2v1_fancy_upsample
        const uint8_t *row = pl + (int64_t)y * pitch;
        const int ix = x >> 1;
        if (!(x & 1)) return ix == 0 ? row[0] : (3 * row[ix] + row[ix - 1] + 1) >> 2;
        return ix == dw - 1 ? row[dw - 1] : (3 * row[ix] + row[ix + 1] + 2) >> 2;
    }
    case UP_H2V2_FANCY: {                                                            // h2v2_fancy_upsample
        const int iy = y >> 1, v = y & 1;
        const int nb = v ? (iy + 1 < dh ? iy + 1 : dh - 1) : (iy > 0 ? iy - 1 : 0);
        const uint8_t *r0 = pl + (int64_t)iy * pitch, *r1 = pl + (int64_t)nb * pitch;
        const int ix = x >> 1;
        const int cs = 3 * r0[ix] + r1[ix];
        if (!(x & 1)) return ix == 0 ? (4 * cs + 8) >> 4 : (3 * cs + 3 * r0[ix - 1] + r1[ix - 1] + 8) >> 4;
        return ix == dw - 1 ? (4 * cs + 7) >> 4 : (3 * cs + 3 * r0[ix + 1] + r1[ix + 1] + 7) >> 4;
    }
    default: return pl[(int64_t)(y / c.vr) * pitch + x / c.hr];                      // h2v1 / h2v2 / int_upsample: replication
    }
}

// ---- colour (jdcolor.c) --------------------------------------------------------------------------------------------------------------
PN_JHD uint8_t clamp255(int v) { return (uint8_t)(v < 0 ? 0 : v > 255 ? 255 : v); }

PN_JHD void ycc_to_bgr(int y, int cb, int cr, uint8_t *bgr) {
    const int64_t xcb = cb - 128, xcr = cr - 128;
    const int r = (int)((91881 * xcr + 32768) >> 16);                    // Cr_r_tab
    const int b = (int)((116130 * xcb + 32768) >> 16);                   // Cb_b_tab
    const int g = (int)((-46802 * xcr + (-22554 * xcb + 32768)) >> 16);  // RIGHT_SHIFT(Cb_g_tab + Cr_g_tab, SCALEBITS)
    bgr[0] = clamp255(y + b);
    bgr[1] = clamp255(y + g);
    bgr[2] = clamp255(y + r);
}

// Pixel (y, x) of the output frame as BGR, from the component planes at scale g (plane[c] has pitch[c] bytes per row).
PN_JHD void pixel_bgr(const pn_jpeg_desc &d, const Scaled &g, const uint8_t *const plane[3], const int pitch[3], int y, int x,
                      uint8_t *bgr) {
    const int Y = upsample(plane[0], pitch[0], g.comp[0], y, x);
    if (d.ncomp == 1) {
        bgr[0] = bgr[1] = bgr[2] = (uint8_t)Y;
        return;
    }
    ycc_to_bgr(Y, upsample(plane[1], pitch[1], g.comp[1], y, x), upsample(plane[2], pitch[2], g.comp[2], y, x), bgr);
}

// The same at full size, for the serial host decoder of tests/test_jpeg_cpu.py: it derives the geometry per pixel, so a loop over
// pixels (csrc/jpeg.cu's color_kernel) calls scaled_geometry once and the overload above.
PN_JHD void pixel_bgr(const pn_jpeg_desc &d, const uint8_t *const plane[3], const int pitch[3], int y, int x, uint8_t *bgr) {
    Scaled g;
    scaled_geometry(d, 1, &g);
    pixel_bgr(d, g, plane, pitch, y, x, bgr);
}

// ---- EXIF orientation (what cv2.imread applies after the decode, at the reduced size too) ------------------------------------------
// o: pn_jpeg_desc.orientation; 0 and 1 are the identity, 2..4 flips, 5..8 transposes (the frame becomes w x h).
PN_JHD bool orient_transposes(int o) { return o >= 5 && o <= 8; }

PN_JHD void oriented_size(int o, int h, int w, int *oh, int *ow) {
    *oh = orient_transposes(o) ? w : h;
    *ow = orient_transposes(o) ? h : w;
}

// Pixel (y, x) of the oriented frame -> pixel (*sy, *sx) of the decoded H x W frame.
PN_JHD void orient_source(int o, int H, int W, int y, int x, int *sy, int *sx) {
    switch (o) {
    case 2: *sy = y; *sx = W - 1 - x; break;                  // flip(1)
    case 3: *sy = H - 1 - y; *sx = W - 1 - x; break;          // flip(-1)
    case 4: *sy = H - 1 - y; *sx = x; break;                  // flip(0)
    case 5: *sy = x; *sx = y; break;                          // transpose
    case 6: *sy = H - 1 - x; *sx = y; break;                  // transpose, flip(1)
    case 7: *sy = H - 1 - x; *sx = W - 1 - y; break;          // transpose, flip(-1)
    case 8: *sy = x; *sx = W - 1 - y; break;                  // transpose, flip(0)
    default: *sy = y; *sx = x;
    }
}

// Where block g (decode order) of an image lands: component and block coordinates in that component's plane.
PN_JHD void block_place(const pn_jpeg_desc &d, int64_t g, int *comp, int *bx, int *by) {
    const int64_t m = g / d.blocks_per_mcu;
    const int b = (int)(g - m * d.blocks_per_mcu);
    const int c = d.mcu_comp[b];
    *comp = c;
    *bx = (int)(m % d.mcus_x) * d.comp[c].h + d.mcu_bx[b];
    *by = (int)(m / d.mcus_x) * d.comp[c].v + d.mcu_by[b];
}

}  // namespace jpeg
}  // namespace pn
