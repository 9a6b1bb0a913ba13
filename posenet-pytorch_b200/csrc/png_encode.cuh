// PNG encode arithmetic, restated from libpng 1.6.53 (pngwutil.c) and zlib 1.3 (deflate.c deflate_rle, trees.c) as cv2 4.13
// calls them for cv2.imencode(".png") without params, as __host__ __device__ functions: csrc/png_enc.cu runs them in parallel,
// tests/test_png_encode_cpu.py compiles them into a serial host encoder and compares its files with cv2 byte for byte.
//
//   filter:    SUB on every row (png_set_filter(PNG_FILTER_SUB)) after png_set_bgr: the byte 0x01, then x[i] - x[i - 3] over the
//              row in RGB order, the first pixel unfiltered.  png_write_start_row drops SUB for an image one pixel wide: the
//              byte 0x00 (NONE) then
//   parse:     deflate_rle at level 1 (Z_BEST_SPEED, Z_RLE, memLevel 8).  Only distance-1 matches exist, so the parse is a
//              closed-form function of the byte runs: a maximal run of length L is one literal, (L - 1) / 258 matches of 258,
//              then the remainder r as one match if r >= 3, else as r literals.  Runs cross rows (the filter bytes are data)
//   blocks:    flushed every lit_bufsize - 1 = 16383 symbols; Z_FINISH always ends with a final block, possibly empty
//   trees:     trees.c build_tree (heap order with the depth tie-break), gen_bitlen (with its overflow fix), gen_codes,
//              build_bl_tree / scan_tree / send_tree, and _tr_flush_block's choice of stored, static or dynamic
//   stored:    only while the block's start is still in the window (block_start >= 0): see slides_before
//   zlib:      windowBits from libpng's png_deflate_claim, the CMF byte rewritten by optimize_cmf, Adler-32 trailer
//   chunks:    signature, IHDR (w, h, 8, 2, 0, 0, 0), IDATs of 8192 bytes but the last, IEND
#pragma once
#include <stdint.h>

#ifdef __CUDACC__
#define PN_PEHD __host__ __device__ __forceinline__
#else
#define PN_PEHD inline
#endif

namespace pn {
namespace pnge {

constexpr int kBlockSyms = 16383;                 // (lit_bufsize - 1) at memLevel 8
constexpr int kIdat = 8192;                       // libpng's PNG_ZBUF_SIZE: the IDAT payload
constexpr int L_CODES = 286, D_CODES = 30, BL_CODES = 19, LITERALS = 256, END_BLOCK = 256;
constexpr int HEAP_SIZE = 2 * L_CODES + 1, MAX_BITS = 15, MAX_BL_BITS = 7;
constexpr int REP_3_6 = 16, REPZ_3_10 = 17, REPZ_11_138 = 18;
constexpr int STORED = 0, STATIC = 1, DYNAMIC = 2;
constexpr int kHeadBytes = 8 + 25;                // signature + IHDR chunk
constexpr int kTailBytes = 12;                    // IEND chunk

// ---- filter and parse --------------------------------------------------------------------------------------------------------
// Byte p of the filtered image (rows of 1 + 3 w bytes) of an h x w BGR frame with rows of 3 w bytes.
PN_PEHD uint8_t filtered_byte(const uint8_t *frame, int w, long long p) {
    const long long rb = 3ll * w + 1;
    const long long r = p / rb;
    const int c = (int)(p - r * rb);
    if (c == 0) return w > 1 ? 1 : 0;
    const int i = c - 1, x = i / 3, ch = 2 - (i - 3 * x);        // RGB order from BGR storage
    const uint8_t *row = frame + r * 3ll * w;
    return (uint8_t)(row[3 * x + ch] - (x ? row[3 * x - 3 + ch] : 0));
}

// Symbols deflate_rle emits for a maximal run of L >= 1 equal bytes.
PN_PEHD long long run_symbols(long long L) {
    const long long q = (L - 1) / 258, r = (L - 1) - 258 * q;
    return 1 + q + (r >= 3 ? 1 : r);
}

// Whether byte j (0 <= j < L) of a run of length L starts a symbol; if so, *lc is its literal (0..255) or 256 + length - 3.
PN_PEHD bool run_symbol_at(long long j, long long L, uint8_t v, int *lc) {
    if (j == 0) { *lc = v; return true; }
    const long long q = (L - 1) / 258, r = (L - 1) - 258 * q;
    const long long m = (j - 1) / 258, o = (j - 1) - 258 * m;
    if (m < q) {
        if (o) return false;
        *lc = 256 + 255;                                          // a match of 258
        return true;
    }
    if (r >= 3) {
        if (o) return false;
        *lc = 256 + (int)r - 3;
        return true;
    }
    *lc = v;                                                      // the literal tail
    return true;
}

// ---- codes -----------------------------------------------------------------------------------------------------------------------
// _length_code[lc] for lc = match length - 3, and its extra bits and base.
PN_PEHD int length_code(int lc) {
    if (lc == 255) return 28;
    if (lc < 8) return lc;
    int b = 3;
    while (lc >> (b + 1)) b++;
    return 4 * (b - 2) + 4 + ((lc >> (b - 2)) & 3);
}
PN_PEHD int length_extra(int code) { return code < 8 || code == 28 ? 0 : (code - 4) >> 2; }
PN_PEHD int length_base(int code) { return code < 8 ? code : code == 28 ? 255 : (4 + (code & 3)) << ((code - 4) >> 2); }

PN_PEHD int lit_extra(int n) { return n > LITERALS ? length_extra(n - LITERALS - 1) : 0; }
PN_PEHD int bl_extra(int n) { return n == REP_3_6 ? 2 : n == REPZ_3_10 ? 3 : n == REPZ_11_138 ? 7 : 0; }

PN_PEHD int static_lit_len(int n) { return n < 144 ? 8 : n < 256 ? 9 : n < 280 ? 7 : 8; }
PN_PEHD int static_lit_canon(int n) { return n < 144 ? 0x30 + n : n < 256 ? 0x190 + n - 144 : n < 280 ? n - 256 : 0xC0 + n - 280; }

PN_PEHD uint32_t bi_reverse(uint32_t code, int len) {
    uint32_t res = 0;
    do {
        res |= code & 1;
        code >>= 1, res <<= 1;
    } while (--len > 0);
    return res >> 1;
}

// ---- trees.c -----------------------------------------------------------------------------------------------------------------------
// One tree (ct_data's Freq / Len / Code kept apart: zlib overlays Dad on Len and Code on Freq).
struct Tree {
    uint16_t *freq, *len, *code;
    int elems, max_code, kind;                    // kind 0 literal / length, 1 distance, 2 bit length
};

struct Scratch {
    int16_t heap[HEAP_SIZE];
    uint8_t depth[HEAP_SIZE];
    uint16_t dad[HEAP_SIZE];
    uint16_t bl_count[MAX_BITS + 1];
    int heap_len, heap_max;
    long long opt_len, static_len;
};

PN_PEHD int tree_extra(const Tree &t, int n) { return t.kind == 0 ? lit_extra(n) : t.kind == 2 ? bl_extra(n) : 0; }
PN_PEHD int tree_static_len(const Tree &t, int n) { return t.kind == 0 ? static_lit_len(n) : 5; }

PN_PEHD bool smaller(const Tree &t, const Scratch &s, int n, int m) {
    return t.freq[n] < t.freq[m] || (t.freq[n] == t.freq[m] && s.depth[n] <= s.depth[m]);
}

PN_PEHD void pqdownheap(const Tree &t, Scratch &s, int k) {
    const int v = s.heap[k];
    int j = k << 1;
    while (j <= s.heap_len) {
        if (j < s.heap_len && smaller(t, s, s.heap[j + 1], s.heap[j])) j++;
        if (smaller(t, s, v, s.heap[j])) break;
        s.heap[k] = s.heap[j];
        k = j;
        j <<= 1;
    }
    s.heap[k] = (int16_t)v;
}

PN_PEHD void gen_bitlen(Tree &t, Scratch &s) {
    const int max_length = t.kind == 2 ? MAX_BL_BITS : MAX_BITS;
    int overflow = 0;
    for (int b = 0; b <= MAX_BITS; b++) s.bl_count[b] = 0;
    t.len[s.heap[s.heap_max]] = 0;                               // the root
    int h;
    for (h = s.heap_max + 1; h < HEAP_SIZE; h++) {
        const int n = s.heap[h];
        int bits = t.len[s.dad[n]] + 1;
        if (bits > max_length) bits = max_length, overflow++;
        t.len[n] = (uint16_t)bits;
        if (n > t.max_code) continue;                             // not a leaf
        s.bl_count[bits]++;
        const int xbits = tree_extra(t, n);
        const long long f = t.freq[n];
        s.opt_len += f * (bits + xbits);
        if (t.kind != 2) s.static_len += f * (tree_static_len(t, n) + xbits);
    }
    if (overflow == 0) return;
    do {
        int bits = max_length - 1;
        while (s.bl_count[bits] == 0) bits--;
        s.bl_count[bits]--;
        s.bl_count[bits + 1] += 2;
        s.bl_count[max_length]--;
        overflow -= 2;
    } while (overflow > 0);
    for (int bits = max_length; bits != 0; bits--) {
        int n = s.bl_count[bits];
        while (n != 0) {
            const int m = s.heap[--h];
            if (m > t.max_code) continue;
            if (t.len[m] != bits) {
                s.opt_len += ((long long)bits - t.len[m]) * t.freq[m];
                t.len[m] = (uint16_t)bits;
            }
            n--;
        }
    }
}

PN_PEHD void gen_codes(Tree &t, const uint16_t *bl_count) {
    uint16_t next_code[MAX_BITS + 1];
    uint32_t code = 0;
    next_code[0] = 0;
    for (int bits = 1; bits <= MAX_BITS; bits++) {
        code = (code + bl_count[bits - 1]) << 1;
        next_code[bits] = (uint16_t)code;
    }
    for (int n = 0; n <= t.max_code; n++) {
        const int len = t.len[n];
        if (len == 0) continue;
        t.code[n] = (uint16_t)bi_reverse(next_code[len]++, len);
    }
}

// build_tree: t.freq[0 .. elems) holds the counts; t.freq / t.len need room for 2 * elems + 1 nodes.
PN_PEHD void build_tree(Tree &t, Scratch &s) {
    int max_code = -1;
    s.heap_len = 0, s.heap_max = HEAP_SIZE;
    for (int n = 0; n < t.elems; n++) {
        if (t.freq[n] != 0) {
            s.heap[++s.heap_len] = (int16_t)(max_code = n);
            s.depth[n] = 0;
        } else {
            t.len[n] = 0;
        }
    }
    while (s.heap_len < 2) {                                      // at least two codes of non-zero frequency
        const int node = s.heap[++s.heap_len] = (int16_t)(max_code < 2 ? ++max_code : 0);
        t.freq[node] = 1;
        s.depth[node] = 0;
        s.opt_len--;
        if (t.kind != 2) s.static_len -= tree_static_len(t, node);
    }
    t.max_code = max_code;
    for (int n = s.heap_len / 2; n >= 1; n--) pqdownheap(t, s, n);
    int node = t.elems;
    do {
        const int n = s.heap[1];                                  // pqremove
        s.heap[1] = s.heap[s.heap_len--];
        pqdownheap(t, s, 1);
        const int m = s.heap[1];
        s.heap[--s.heap_max] = (int16_t)n;
        s.heap[--s.heap_max] = (int16_t)m;
        t.freq[node] = (uint16_t)(t.freq[n] + t.freq[m]);
        s.depth[node] = (uint8_t)((s.depth[n] >= s.depth[m] ? s.depth[n] : s.depth[m]) + 1);
        s.dad[n] = s.dad[m] = (uint16_t)node;
        s.heap[1] = (int16_t)node++;
        pqdownheap(t, s, 1);
    } while (s.heap_len >= 2);
    s.heap[--s.heap_max] = s.heap[1];
    gen_bitlen(t, s);
    gen_codes(t, s.bl_count);
}

// scan_tree / send_tree walk the code lengths 0 .. max_code; the length past max_code reads as zlib's 0xffff guard.
PN_PEHD int len_or_guard(const uint16_t *len, int n, int max_code) { return n > max_code ? 0xffff : len[n]; }

template <typename Visit>
PN_PEHD void walk_tree(const uint16_t *len, int max_code, Visit &&visit) {
    int prevlen = -1, nextlen = len_or_guard(len, 0, max_code), count = 0, max_count = 7, min_count = 4;
    if (nextlen == 0) max_count = 138, min_count = 3;
    for (int n = 0; n <= max_code; n++) {
        const int curlen = nextlen;
        nextlen = len_or_guard(len, n + 1, max_code);
        if (++count < max_count && curlen == nextlen) continue;
        visit(curlen, count, prevlen, min_count);
        count = 0;
        prevlen = curlen;
        if (nextlen == 0) max_count = 138, min_count = 3;
        else if (curlen == nextlen) max_count = 6, min_count = 3;
        else max_count = 7, min_count = 4;
    }
}

PN_PEHD void scan_tree(const uint16_t *len, int max_code, uint16_t *bl_freq) {
    walk_tree(len, max_code, [&](int curlen, int count, int prevlen, int min_count) {
        if (count < min_count) bl_freq[curlen] += count;
        else if (curlen != 0) {
            if (curlen != prevlen) bl_freq[curlen]++;
            bl_freq[REP_3_6]++;
        } else if (count <= 10) bl_freq[REPZ_3_10]++;
        else bl_freq[REPZ_11_138]++;
    });
}

template <typename Sink>
PN_PEHD void send_tree(const uint16_t *len, int max_code, const uint16_t *bl_code, const uint16_t *bl_len, Sink &out) {
    walk_tree(len, max_code, [&](int curlen, int count, int prevlen, int min_count) {
        if (count < min_count) {
            do { out(bl_code[curlen], bl_len[curlen]); } while (--count != 0);
        } else if (curlen != 0) {
            if (curlen != prevlen) {
                out(bl_code[curlen], bl_len[curlen]);
                count--;
            }
            out(bl_code[REP_3_6], bl_len[REP_3_6]);
            out(count - 3, 2);
        } else if (count <= 10) {
            out(bl_code[REPZ_3_10], bl_len[REPZ_3_10]);
            out(count - 3, 3);
        } else {
            out(bl_code[REPZ_11_138], bl_len[REPZ_11_138]);
            out(count - 11, 7);
        }
    });
}

PN_PEHD int bl_order(int k) {                                    // {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15}
    switch (k) {
    case 0: return 16; case 1: return 17; case 2: return 18; case 3: return 0; case 4: return 8; case 5: return 7;
    case 6: return 9; case 7: return 6; case 8: return 10; case 9: return 5; case 10: return 11; case 11: return 4;
    case 12: return 12; case 13: return 3; case 14: return 13; case 15: return 2; case 16: return 14; case 17: return 1;
    default: return 15;
    }
}

// Everything the bit writer needs for one block.
struct BlockCode {
    uint16_t code[L_CODES];                       // literal / length codes (bit-reversed, as send_bits takes them)
    uint8_t len[L_CODES];
    uint16_t bl_code[BL_CODES];
    uint8_t bl_len[BL_CODES];
    int type, lcodes, blcodes, dlen;              // dlen: the length of distance code 0, the only one Z_RLE uses
    long long bits;                               // static / dynamic: the block's bits from its 3-bit type on
};

// The storage _tr_flush_block works in: three trees and the heap.
struct FlushWork {
    uint16_t lfreq[HEAP_SIZE], llen[HEAP_SIZE], lcode[L_CODES];
    uint16_t dfreq[2 * D_CODES + 1], dlen[2 * D_CODES + 1], dcode[D_CODES];
    uint16_t bfreq[2 * BL_CODES + 1], blen[2 * BL_CODES + 1], bcode[BL_CODES];
    Scratch s;
};

// _tr_flush_block's trees and choice.  lit_freq[0 .. 286): the block's literal / length counts without END_BLOCK; matches: the
// number of matches (all at distance 1); stored_len: the block's bytes; storable: block_start >= 0.
PN_PEHD void flush_block(const uint32_t *lit_freq, uint32_t matches, long long stored_len, bool storable, FlushWork &w,
                         BlockCode *out) {
    for (int n = 0; n < L_CODES; n++) w.lfreq[n] = (uint16_t)lit_freq[n];
    w.lfreq[END_BLOCK] = 1;
    for (int n = 0; n < D_CODES; n++) w.dfreq[n] = 0;
    w.dfreq[0] = (uint16_t)matches;
    for (int n = 0; n < BL_CODES; n++) w.bfreq[n] = 0;
    w.s.opt_len = w.s.static_len = 0;
    Tree lt{w.lfreq, w.llen, w.lcode, L_CODES, 0, 0}, dt{w.dfreq, w.dlen, w.dcode, D_CODES, 0, 1},
        bt{w.bfreq, w.blen, w.bcode, BL_CODES, 0, 2};
    build_tree(lt, w.s);
    build_tree(dt, w.s);
    scan_tree(w.llen, lt.max_code, w.bfreq);                      // build_bl_tree
    scan_tree(w.dlen, dt.max_code, w.bfreq);
    build_tree(bt, w.s);
    int max_blindex;
    for (max_blindex = BL_CODES - 1; max_blindex >= 3; max_blindex--)
        if (w.blen[bl_order(max_blindex)] != 0) break;
    w.s.opt_len += 3 * ((long long)max_blindex + 1) + 5 + 5 + 4;
    long long opt_lenb = (w.s.opt_len + 3 + 7) >> 3;
    const long long static_lenb = (w.s.static_len + 3 + 7) >> 3;
    if (static_lenb <= opt_lenb) opt_lenb = static_lenb;
    if (stored_len + 4 <= opt_lenb && storable) {
        out->type = STORED;
        out->bits = 0;
        return;
    }
    if (static_lenb == opt_lenb) {
        out->type = STATIC;
        out->bits = 3 + w.s.static_len;
        for (int n = 0; n < L_CODES; n++) {
            out->len[n] = (uint8_t)static_lit_len(n);
            out->code[n] = (uint16_t)bi_reverse(static_lit_canon(n), static_lit_len(n));
        }
        out->dlen = 5;
        return;
    }
    out->type = DYNAMIC;
    out->bits = 3 + w.s.opt_len;
    for (int n = 0; n < L_CODES; n++) {
        out->len[n] = (uint8_t)(n <= lt.max_code ? w.llen[n] : 0);
        out->code[n] = n <= lt.max_code ? w.lcode[n] : 0;
    }
    for (int n = 0; n < BL_CODES; n++) {
        out->bl_len[n] = (uint8_t)w.blen[n];
        out->bl_code[n] = w.bcode[n];
    }
    out->lcodes = lt.max_code + 1;
    out->blcodes = max_blindex + 1;
    out->dlen = w.dlen[0];                                        // the distance tree is always lengths 1, 1
}

// The bits of one symbol under a block's codes.
PN_PEHD int symbol_bits(const BlockCode &b, int lc) {
    if (lc < 256) return b.len[lc];
    const int code = length_code(lc - 256);
    return b.len[code + LITERALS + 1] + length_extra(code) + b.dlen;
}

// ---- the bit writer (send_bits: LSB first) ------------------------------------------------------------------------------------
template <typename Sink>
PN_PEHD void send_symbol(const BlockCode &b, int lc, Sink &out) {
    if (lc < 256) {
        out(b.code[lc], b.len[lc]);
        return;
    }
    const int l = lc - 256, code = length_code(l);
    out(b.code[code + LITERALS + 1], b.len[code + LITERALS + 1]);
    const int e = length_extra(code);
    if (e) out(l - length_base(code), e);
    out(0u, b.dlen);                                              // distance code 0 is all zero bits, static or dynamic
}

// The 3-bit block type and, for a dynamic block, send_all_trees (the literal tree from its lengths; the distance tree is
// always two codes of length 1).
template <typename Sink>
PN_PEHD void send_block_header(const BlockCode &b, bool last, Sink &out) {
    out((uint32_t)((b.type == DYNAMIC ? 2 : b.type == STATIC ? 1 : 0) << 1) + (last ? 1 : 0), 3);
    if (b.type != DYNAMIC) return;
    out(b.lcodes - 257, 5);
    out(2 - 1, 5);
    out(b.blcodes - 4, 4);
    for (int rank = 0; rank < b.blcodes; rank++) out(b.bl_len[bl_order(rank)], 3);
    uint16_t llen[L_CODES], blc[BL_CODES], bll[BL_CODES];
    for (int n = 0; n < L_CODES; n++) llen[n] = b.len[n];
    for (int n = 0; n < BL_CODES; n++) blc[n] = b.bl_code[n], bll[n] = b.bl_len[n];
    send_tree(llen, b.lcodes - 1, blc, bll, out);
    const uint16_t dl[2] = {1, 1};
    send_tree(dl, 1, blc, bll, out);
}

// Header bits of a dynamic block (0 otherwise) beyond the 3-bit type.
struct CountBits {
    long long bits = 0;
    PN_PEHD void operator()(uint32_t, int n) { bits += n; }
};

// ---- the window: which blocks may be stored ---------------------------------------------------------------------------------
// Number of window slides (fill_window moving the upper half down by w = 2^wbits bytes) deflate_rle has made when it flushes a
// block whose last symbol starts at byte p of an n-byte input (p = n for the final block).  Slide j (j >= 1) happens at the
// first loop top at or past T_j = max((j + 1) w - 262, min(n, (j + 1) w) - 258): with all the input at hand the lookahead only
// drops to MAX_MATCH there.  A block starting at byte b is stored only if b >= slides * w.  (An input fed row by row, as
// libpng does, can slide up to four bytes earlier; a block that this changes spans more than w - 262 bytes with at most 16383
// symbols, and such a block never codes larger than it is, so the stored choice is the same.)
PN_PEHD long long slides_before(long long p, long long n, int wbits) {
    const long long w = 1ll << wbits;
    const long long full = n / w;                                 // multiples m = j + 1 with m w <= n
    long long k = 0;
    const long long a = (p + 258) / w < full ? (p + 258) / w : full;
    if (a >= 2) k += a - 1;
    if (n - 258 <= p) {                                           // at most one multiple past n within reach
        const long long lo = full + 1 > 2 ? full + 1 : 2, hi = (p + 262) / w;
        if (hi >= lo) k += hi - lo + 1;
    }
    return k;
}

// ---- zlib and PNG framing ----------------------------------------------------------------------------------------------------
// png_deflate_claim's windowBits for the filtered image size.
PN_PEHD int window_bits(long long data_size) {
    int wb = 15;
    if (data_size <= 16384) {
        unsigned half = 1u << (wb - 1);
        while (data_size + 262 <= half) {
            half >>= 1;
            --wb;
        }
    }
    return wb;
}

// The zlib header (level 1, Z_RLE: FLEVEL 0), then libpng's optimize_cmf.
PN_PEHD void zlib_header(long long data_size, int wbits, uint8_t *h) {
    unsigned cmf = 0x08 | ((wbits - 8) << 4), hdr = cmf << 8;
    hdr += 31 - hdr % 31;
    unsigned flg = hdr & 0xFF;
    if (data_size <= 16384 && (cmf & 0xF0) <= 0x70) {
        unsigned cinfo = cmf >> 4, half = 1u << (cinfo + 7);
        if (data_size <= half) {
            do {
                half >>= 1;
                --cinfo;
            } while (cinfo > 0 && data_size <= half);
            cmf = (cmf & 0x0F) | (cinfo << 4);
            unsigned tmp = flg & 0xE0;
            tmp += 0x1F - ((cmf << 8) + tmp) % 0x1F;
            flg = tmp;
        }
    }
    h[0] = (uint8_t)cmf;
    h[1] = (uint8_t)flg;
}

constexpr uint32_t kAdlerBase = 65521;
constexpr uint32_t kCrcPoly = 0xEDB88320u;

PN_PEHD uint32_t crc32_update(uint32_t crc, const uint8_t *p, long long n) {    // standard CRC-32, bitwise
    crc = ~crc;
    for (long long i = 0; i < n; i++) {
        crc ^= p[i];
        for (int k = 0; k < 8; k++) crc = crc & 1 ? (crc >> 1) ^ kCrcPoly : crc >> 1;
    }
    return ~crc;
}

// zlib's multmodp / x2nmodp / crc32_combine: crc(A || B) from crc(A), crc(B) and |B|.
PN_PEHD uint32_t multmodp(uint32_t a, uint32_t b) {
    uint32_t m = 1u << 31, p = 0;
    for (;;) {
        if (a & m) {
            p ^= b;
            if ((a & (m - 1)) == 0) break;
        }
        m >>= 1;
        b = b & 1 ? (b >> 1) ^ kCrcPoly : b >> 1;
    }
    return p;
}
PN_PEHD uint32_t crc32_combine(uint32_t crc1, uint32_t crc2, long long len2) {
    uint32_t p = 1u << 31, x2n = 1u << 30;                       // x^0, x^(2^0)
    for (int k = 0; k < 3; k++) x2n = multmodp(x2n, x2n);        // x^(2^3): one byte
    for (long long n = len2; n; n >>= 1) {
        if (n & 1) p = multmodp(x2n, p);
        x2n = multmodp(x2n, x2n);
    }
    return multmodp(p, crc1) ^ crc2;
}

PN_PEHD void put_be32(uint8_t *o, uint32_t v) {
    o[0] = (uint8_t)(v >> 24), o[1] = (uint8_t)(v >> 16), o[2] = (uint8_t)(v >> 8), o[3] = (uint8_t)v;
}

// Signature and IHDR chunk (33 bytes) of an h x w RGB image.
PN_PEHD void write_head(int h, int w, uint8_t *o) {
    const uint8_t sig[8] = {0x89, 'P', 'N', 'G', 0x0D, 0x0A, 0x1A, 0x0A};
    for (int k = 0; k < 8; k++) o[k] = sig[k];
    put_be32(o + 8, 13);
    o[12] = 'I', o[13] = 'H', o[14] = 'D', o[15] = 'R';
    put_be32(o + 16, (uint32_t)w);
    put_be32(o + 20, (uint32_t)h);
    o[24] = 8, o[25] = 2, o[26] = 0, o[27] = 0, o[28] = 0;
    put_be32(o + 29, crc32_update(0, o + 12, 17));
}

PN_PEHD void write_tail(uint8_t *o) {
    const uint8_t iend[12] = {0, 0, 0, 0, 'I', 'E', 'N', 'D', 0xAE, 0x42, 0x60, 0x82};
    for (int k = 0; k < 12; k++) o[k] = iend[k];
}

PN_PEHD long long num_chunks(long long zlen) { return (zlen + kIdat - 1) / kIdat; }
PN_PEHD long long file_size(long long zlen) { return kHeadBytes + zlen + 12 * num_chunks(zlen) + kTailBytes; }

// Filtered bytes of an h x w frame.
PN_PEHD long long data_size(int h, int w) { return (long long)h * (3ll * w + 1); }

// Most blocks an n-byte input can make (symbols <= bytes), the final one included.
PN_PEHD long long max_blocks(long long n) { return n / kBlockSyms + 1; }

// A true worst case of the deflate stream: a block of len bytes that is not stored costs at most its static coding, 3 + 9 len
// + 7 bits (a literal at most 9 bits, a match of L >= 3 bytes at most 8 + 5 + 5); a stored block is only chosen when its
// len + 4 bytes fit in that coding rounded up to bytes, so it costs at most 9 len + 27 bits with its type and alignment.
PN_PEHD long long deflate_bound(long long n) { return (9 * n + 32 * max_blocks(n) + 7) / 8 + 1; }
PN_PEHD long long zlib_bound(long long n) { return 2 + deflate_bound(n) + 4; }
PN_PEHD long long encode_bound(int h, int w) { return h && w ? file_size(zlib_bound(data_size(h, w))) : 0; }

}  // namespace pnge
}  // namespace pn
