// Progressive JPEG entropy decode, restated from libjpeg-turbo 3.1's jdphuff.c (what cv2 4.13 runs for a progressive file), as
// __host__ __device__ functions: csrc/jpeg.cu runs one restart segment of one scan per thread, tests/test_jpeg_progressive_cpu.py
// compiles them into a serial host decoder and compares it with cv2 byte for byte.
//
//   bit reader:  jpeg_fill_bit_buffer over the raw file bytes: 0xFF 0x00 is a data 0xFF, 0xFF fill bytes collapse, a marker or the
//                end of the segment ends the data and zeros are read past it
//   decoders:    decode_mcu_DC_first, decode_mcu_DC_refine, decode_mcu_AC_first (EOBRUN) and decode_mcu_AC_refine (correction
//                bits, p1 / m1), storing into the coefficient array that the baseline IDCT reads, in the descriptor's
//                interleaved block order (block_place)
// Where libjpeg warns (a bad Huffman code, data needed past the segment's end, more than 7 bits left over, a refinement symbol of
// size other than 1) the segment fails.  A run that would store a coefficient outside the scan's band (libjpeg stores it at
// jpeg_natural_order[k]) fails too: the scans of one wave run in parallel on disjoint bands.
#pragma once
#include "jpeg_decode.cuh"

namespace pn {
namespace jpeg {

// ---- the scan table (pn_jpeg_parse_progressive), at file_offset + align8(file_bytes) in the byte arena ---------------------------
PN_JHD int64_t scan_table_bytes(int n_scans, int n_huff) {
    return (int64_t)sizeof(pn_jpeg_scans) + (int64_t)n_scans * sizeof(pn_jpeg_scan) + (int64_t)n_huff * sizeof(pn_jpeg_huff);
}
PN_JHD int64_t scan_table_offset(const pn_jpeg_desc &d) { return d.file_offset + ((d.file_bytes + 7) & ~(int64_t)7); }
PN_JHD const pn_jpeg_scan *table_scans(const uint8_t *t) { return reinterpret_cast<const pn_jpeg_scan *>(t + sizeof(pn_jpeg_scans)); }
PN_JHD const pn_jpeg_huff *table_huff(const uint8_t *t) {
    const int n = reinterpret_cast<const pn_jpeg_scans *>(t)->n_scans;
    return reinterpret_cast<const pn_jpeg_huff *>(t + sizeof(pn_jpeg_scans) + sizeof(pn_jpeg_scan) * n);
}

// ---- scan geometry (jdinput.c per_scan_setup) ---------------------------------------------------------------------------------
// Units: MCUs of an interleaved scan (the frame's MCU grid), blocks of the component's own grid in a one-component scan.
PN_JHD int scan_units_x(const pn_jpeg_desc &d, const pn_jpeg_scan &s) {
    return s.ncomp > 1 ? d.mcus_x : (d.comp[s.comp[0]].dw + 7) / 8;
}
PN_JHD int64_t scan_units(const pn_jpeg_desc &d, const pn_jpeg_scan &s) {
    return s.ncomp > 1 ? (int64_t)d.mcus_x * d.mcus_y : (int64_t)scan_units_x(d, s) * ((d.comp[s.comp[0]].dh + 7) / 8);
}
PN_JHD int64_t scan_segments(const pn_jpeg_desc &d, const pn_jpeg_scan &s) {
    const int64_t u = scan_units(d, s);
    return s.restart_interval > 0 ? (u + s.restart_interval - 1) / s.restart_interval : 1;
}

// The MCU layout pn_jpeg_parse_progressive gives a kind-2 descriptor, which coef_block relies on: every component in frame
// order, its h x v blocks in raster order (one component: a single 1 x 1 block).  plan_kernel rejects any other layout.
PN_JHD bool canonical_mcu(const pn_jpeg_desc &d) {
    if (d.ncomp < 1 || d.ncomp > 3 || (d.ncomp == 1 && (d.comp[0].h != 1 || d.comp[0].v != 1))) return false;
    int nb = 0;
    for (int c = 0; c < d.ncomp; ++c)
        for (int by = 0; by < d.comp[c].v; ++by)
            for (int bx = 0; bx < d.comp[c].h; ++bx, ++nb)
                if (nb >= PN_JPEG_MAX_BLOCKS || d.mcu_comp[nb] != c || d.mcu_bx[nb] != bx || d.mcu_by[nb] != by) return false;
    return nb == d.blocks_per_mcu;
}

// Block (bx, by) of component c in the coefficient array of a canonical_mcu descriptor: the inverse of block_place.
PN_JHD int64_t coef_block(const pn_jpeg_desc &d, int c, int bx, int by) {
    int first = 0;                      // the component's first block in the MCU
    for (int k = 0; k < c; ++k) first += d.comp[k].h * d.comp[k].v;
    const pn_jpeg_comp &k = d.comp[c];
    const int64_t m = (int64_t)(by / k.v) * d.mcus_x + bx / k.h;
    return m * d.blocks_per_mcu + first + (by % k.v) * k.h + bx % k.h;
}

// First RSTn marker (0xFF 0xD0..0xD7) at or after p in [p, end): its 0xFF, or end.
PN_JHD int64_t next_restart(const uint8_t *f, int64_t p, int64_t end) {
    for (int64_t q = p; q + 1 < end; ++q)
        if (f[q] == 0xFF && (f[q + 1] & 0xF8) == 0xD0) return q;
    return end;
}

// ---- bit reader over one segment's raw bytes [pos, end) ---------------------------------------------------------------------------
struct ScanBits {
    const uint8_t *f;
    int64_t pos, end;
    int64_t stop;     // where the data ended (a marker's 0xFF, or end); -1 before
    uint64_t acc;     // MSB first
    int n, zeros;     // bits in acc; of those, the zero bits inserted past the data (always the last ones)

    PN_JHD ScanBits(const uint8_t *file, int64_t start, int64_t e) : f(file), pos(start), end(e), stop(-1), acc(0), n(0), zeros(0) {}
    PN_JHD void fill() {
        while (n <= 56) {
            uint32_t c = 0;
            if (stop < 0) {
                if (pos >= end) {
                    stop = end;
                } else if ((c = f[pos++]) == 0xFF) {
                    while (pos < end && f[pos] == 0xFF) ++pos;
                    if (pos < end && f[pos] == 0) {
                        ++pos;
                    } else {
                        stop = pos < end ? pos - 1 : end;
                        c = 0;
                    }
                }
            }
            if (stop >= 0) zeros += 8;
            acc |= (uint64_t)c << (56 - n);
            n += 8;
        }
    }
    PN_JHD uint32_t peek32() {
        if (n < 32) fill();
        return (uint32_t)(acc >> 32);
    }
    PN_JHD void skip(int k) {
        acc <<= k;
        n -= k;
    }
    PN_JHD uint32_t get(int k) {                // k in 1..16
        const uint32_t v = peek32() >> (32 - k);
        skip(k);
        return v;
    }
    PN_JHD int symbol(const pn_jpeg_huff &t) {  // HUFF_DECODE; -1 for a code not in the table
        int sym;
        const int len = huff_symbol(t, peek32(), &sym);
        if (!len) return -1;
        skip(len);
        return sym;
    }
    // After a segment's last unit: no bit was taken past the data, the data ended at `end`, at most 7 bits are left over.
    PN_JHD int finish() {
        if (n < zeros) return PN_JPEG_ERR_LENGTH;
        fill();
        if (stop != end) return PN_JPEG_ERR_RESTART;
        return n - zeros > 7 ? PN_JPEG_ERR_LENGTH : PN_JPEG_OK;
    }
};

PN_JHD int16_t jcoef(int v) { return (int16_t)(uint16_t)(uint32_t)v; }       // (JCOEF) of an int

// ---- one restart segment of one scan: units [u0, u0 + nu) from the bytes [start, end) ----------------------------------------------
// coef: the image's coefficient array (zeroed before its first scan).  Returns PN_JPEG_OK or a status < 0.
PN_JHD int decode_scan_segment(const pn_jpeg_desc &d, const pn_jpeg_scan &S, const pn_jpeg_huff *huff, const uint8_t *file,
                               int64_t start, int64_t end, int64_t u0, int64_t nu, int16_t *coef) {
    ScanBits r(file, start, end);
    const int al = S.al, ss = S.ss, se = S.se;
    const int p1 = 1 << al, m1 = (int)(~0u << al);
    const int ux = scan_units_x(d, S);
    int last_dc[3] = {0, 0, 0};
    uint32_t eobrun = 0;
    for (int64_t u = u0; u < u0 + nu; ++u) {
        if (S.ncomp == 1) {
            const int c = S.comp[0];
            int16_t *blk = coef + coef_block(d, c, (int)(u % ux), (int)(u / ux)) * 64;
            if (ss == 0) {
                if (S.ah) {                                                  // decode_mcu_DC_refine
                    if (r.get(1)) blk[0] = jcoef(blk[0] | p1);
                } else {                                                     // decode_mcu_DC_first
                    const int s = r.symbol(huff[S.dc[0]]);
                    if (s < 0) return PN_JPEG_ERR_CODE;
                    const int diff = s ? huff_extend(r.get(s), s) : 0;
                    if ((last_dc[0] >= 0 && diff > 0x7FFFFFFF - last_dc[0]) || (last_dc[0] < 0 && diff < (-0x7FFFFFFF - 1) - last_dc[0]))
                        return PN_JPEG_ERR_CODE;                             // JERR_BAD_DCT_COEF
                    last_dc[0] += diff;
                    blk[0] = jcoef((int)((uint32_t)last_dc[0] << al));
                }
            } else if (S.ah == 0) {                                          // decode_mcu_AC_first
                if (eobrun > 0) {
                    --eobrun;
                    continue;
                }
                const pn_jpeg_huff &t = huff[S.ac[0]];
                for (int k = ss; k <= se; ++k) {
                    const int sym = r.symbol(t);
                    if (sym < 0) return PN_JPEG_ERR_CODE;
                    int rr = sym >> 4;
                    const int s = sym & 15;
                    if (s) {
                        k += rr;
                        if (k > se) return PN_JPEG_ERR_CODE;
                        blk[natural_order(k)] = jcoef((int)((uint32_t)huff_extend(r.get(s), s) << al));
                    } else if (rr == 15) {
                        k += 15;
                    } else {
                        eobrun = 1u << rr;
                        if (rr) eobrun += r.get(rr);
                        --eobrun;
                        break;
                    }
                }
            } else {                                                         // decode_mcu_AC_refine
                const pn_jpeg_huff &t = huff[S.ac[0]];
                int k = ss;
                if (eobrun == 0) {
                    for (; k <= se; ++k) {
                        const int sym = r.symbol(t);
                        if (sym < 0) return PN_JPEG_ERR_CODE;
                        int rr = sym >> 4, s = sym & 15;
                        if (s) {
                            if (s != 1) return PN_JPEG_ERR_CODE;             // JWRN_HUFF_BAD_CODE
                            s = r.get(1) ? p1 : m1;
                        } else if (rr != 15) {
                            eobrun = 1u << rr;
                            if (rr) eobrun += r.get(rr);
                            break;                                           // the rest of the block: the EOB logic below
                        }
                        do {                                                 // correction bits up to the rr+1-th zero coefficient
                            int16_t &x = blk[natural_order(k)];
                            if (x != 0) {
                                if (r.get(1) && (x & p1) == 0) x = jcoef(x >= 0 ? x + p1 : x + m1);
                            } else if (--rr < 0) {
                                break;
                            }
                            ++k;
                        } while (k <= se);
                        if (s) {
                            if (k > se) return PN_JPEG_ERR_CODE;
                            blk[natural_order(k)] = jcoef(s);
                        }
                    }
                }
                if (eobrun > 0) {
                    for (; k <= se; ++k) {
                        int16_t &x = blk[natural_order(k)];
                        if (x != 0 && r.get(1) && (x & p1) == 0) x = jcoef(x >= 0 ? x + p1 : x + m1);
                    }
                    --eobrun;
                }
            }
            continue;
        }
        // an interleaved DC scan: every block of the MCU, components in scan order
        const int64_t mx = u % d.mcus_x, my = u / d.mcus_x;
        for (int i = 0; i < S.ncomp; ++i) {
            const int c = S.comp[i];
            const pn_jpeg_comp &k = d.comp[c];
            for (int y = 0; y < k.v; ++y)
                for (int x = 0; x < k.h; ++x) {
                    int16_t *blk = coef + coef_block(d, c, (int)(mx * k.h + x), (int)(my * k.v + y)) * 64;
                    if (S.ah) {
                        if (r.get(1)) blk[0] = jcoef(blk[0] | p1);
                        continue;
                    }
                    const int s = r.symbol(huff[S.dc[i]]);
                    if (s < 0) return PN_JPEG_ERR_CODE;
                    const int diff = s ? huff_extend(r.get(s), s) : 0;
                    if ((last_dc[i] >= 0 && diff > 0x7FFFFFFF - last_dc[i]) || (last_dc[i] < 0 && diff < (-0x7FFFFFFF - 1) - last_dc[i]))
                        return PN_JPEG_ERR_CODE;
                    last_dc[i] += diff;
                    blk[0] = jcoef((int)((uint32_t)last_dc[i] << al));
                }
        }
    }
    return r.finish();
}

}  // namespace jpeg
}  // namespace pn
