// pn_jpeg_parse: the header walk of libjpeg-turbo's jdmarker.c / jdinput.c for the files csrc/jpeg.cu decodes, in host code (no
// device needed).  Everything that would make libjpeg-turbo (or cv2 around it) do something other than a plain baseline decode --
// progressive or arithmetic coding, other precisions, several scans, CMYK / RGB colour, EXIF rotation, a warning -- classifies the
// file PN_JPEG_HOST, so that the GPU path only ever decodes files cv2 reads without comment.  pn_jpeg_parse_oriented also accepts
// files whose EXIF rotation is certain (read_exif) and records it for the decode to apply.  pn_jpeg_parse_progressive also
// accepts progressive files with a complete, warning-free scan script, walking every scan into a scan table (progressive_scan).
#include <string.h>

#include "common.cuh"
#include "jpeg_decode.cuh"
#include "jpeg_progressive.cuh"

namespace pn {
namespace {

struct Reader {
    const uint8_t *f;
    int64_t n;
    int u8(int64_t p) const { return p < n ? f[p] : -1; }
    int u16(int64_t p) const { return p + 1 < n ? (f[p] << 8) | f[p + 1] : -1; }
};

int host(pn_jpeg_desc *d, int why) {
    d->kind = PN_JPEG_HOST;
    d->why = why;
    return PN_OK;
}

// jpeg_make_d_derived_tbl, with its validation.  false: the table is invalid (libjpeg: JERR_BAD_HUFF_TABLE).
bool derive(const uint8_t bits[17], const uint8_t *vals, bool is_dc, pn_jpeg_huff *t) {
    memset(t, 0, sizeof(*t));
    char size[257];
    unsigned code_of[257];
    int p = 0;
    for (int l = 1; l <= 16; ++l) {
        const int i = bits[l];
        if (p + i > 256) return false;
        for (int k = 0; k < i; ++k) size[p++] = (char)l;
    }
    size[p] = 0;
    const int nsym = p;
    unsigned code = 0;
    int si = size[0];
    p = 0;
    while (size[p]) {
        while (size[p] == si) {
            code_of[p++] = code;
            ++code;
        }
        if (code >= (1u << si)) return false;
        code <<= 1;
        ++si;
    }
    p = 0;
    for (int l = 1; l <= 16; ++l) {
        if (bits[l]) {
            t->valoffset[l] = p - (int32_t)code_of[p];
            p += bits[l];
            t->maxcode[l] = (int32_t)code_of[p - 1];
        } else {
            t->maxcode[l] = -1;
        }
    }
    t->valoffset[17] = 0;
    t->maxcode[17] = 0xFFFFF;
    p = 0;
    for (int l = 1; l <= 8; ++l)
        for (int i = 1; i <= bits[l]; ++i, ++p) {
            const int look = (int)(code_of[p] << (8 - l));
            for (int ctr = 1 << (8 - l); ctr > 0; --ctr) t->lookup[look + ctr - 1] = (uint16_t)((l << 8) | vals[p]);
        }
    for (int i = 0; i < nsym; ++i) {
        t->huffval[i] = vals[i];
        if (is_dc && vals[i] > 15) return false;
    }
    return true;
}

// Geometry of a scan of the ns components order[0..ns) (jdinput.c initial_setup / per_scan_setup) into the descriptor: planes,
// MCU grid and the blocks of one MCU.  false: sampling factors libjpeg rejects.
bool geometry(pn_jpeg_desc *d, const int *comp_h, const int *comp_v, const int *order, int ns) {
    int max_h = 1, max_v = 1;
    for (int c = 0; c < d->ncomp; ++c) {
        max_h = comp_h[c] > max_h ? comp_h[c] : max_h;
        max_v = comp_v[c] > max_v ? comp_v[c] : max_v;
    }
    for (int c = 0; c < d->ncomp; ++c) {
        if (max_h % comp_h[c] || max_v % comp_v[c]) return false;
        pn_jpeg_comp &k = d->comp[c];
        k.hr = max_h / comp_h[c];
        k.vr = max_v / comp_v[c];
        k.dw = (int)(((int64_t)d->width * comp_h[c] + max_h - 1) / max_h);
        k.dh = (int)(((int64_t)d->height * comp_v[c] + max_v - 1) / max_v);
    }
    if (ns == 1) {                       // non-interleaved: one block per MCU over the component's own block grid
        pn_jpeg_comp &k = d->comp[0];
        k.h = k.v = 1;
        d->mcus_x = k.bw = (k.dw + 7) / 8;
        d->mcus_y = k.bh = (k.dh + 7) / 8;
        d->blocks_per_mcu = 1;
        d->mcu_comp[0] = 0;
    } else {
        d->mcus_x = (d->width + 8 * max_h - 1) / (8 * max_h);
        d->mcus_y = (d->height + 8 * max_v - 1) / (8 * max_v);
        int nb = 0;
        for (int s = 0; s < ns; ++s) {
            const int c = order[s];
            pn_jpeg_comp &k = d->comp[c];
            k.h = comp_h[c];
            k.v = comp_v[c];
            k.bw = d->mcus_x * k.h;
            k.bh = d->mcus_y * k.v;
            if (nb + k.h * k.v > PN_JPEG_MAX_BLOCKS) return false;
            for (int by = 0; by < k.v; ++by)
                for (int bx = 0; bx < k.h; ++bx, ++nb) {
                    d->mcu_comp[nb] = (uint8_t)c;
                    d->mcu_bx[nb] = (uint8_t)bx;
                    d->mcu_by[nb] = (uint8_t)by;
                }
        }
        d->blocks_per_mcu = nb;
    }
    return true;
}

// What one APP1 "Exif\0\0" payload says about the orientation (tag 0x0112 of IFD0).
struct Exif {
    bool readable;   // II / MM, 42, IFD0 and all of its entries inside the payload
    int tags;        // 0x0112 entries in IFD0
    int value;       // the first one's value (SHORT), 0 when it has another type; 1 without the tag
    bool strict;     // every 0x0112 entry is a SHORT with count 1, and cv2 reads up to it (below)
};

// Bytes of a TIFF field type (1..12), 0 for an unknown type.
int type_bytes(int type) {
    static const int kBytes[13] = {0, 1, 1, 2, 4, 8, 1, 1, 2, 4, 8, 4, 8};
    return type >= 1 && type <= 12 ? kBytes[type] : 0;
}

Exif read_exif(const uint8_t *p, int64_t n) {
    Exif e{false, 0, 1, true};
    if (n < 14) return e;
    const uint8_t *t = p + 6;
    const int64_t tn = n - 6;
    bool le;
    if (t[0] == 'I' && t[1] == 'I') le = true;
    else if (t[0] == 'M' && t[1] == 'M') le = false;
    else return e;
    auto r16 = [&](int64_t o) -> int { return le ? t[o] | (t[o + 1] << 8) : (t[o] << 8) | t[o + 1]; };
    auto r32 = [&](int64_t o) -> int64_t {
        return le ? (int64_t)t[o] | ((int64_t)t[o + 1] << 8) | ((int64_t)t[o + 2] << 16) | ((int64_t)t[o + 3] << 24)
                  : ((int64_t)t[o] << 24) | ((int64_t)t[o + 1] << 16) | ((int64_t)t[o + 2] << 8) | (int64_t)t[o + 3];
    };
    if (r16(2) != 42) return e;
    const int64_t ifd = r32(4);
    if (ifd < 8 || ifd + 2 > tn) return e;
    const int cnt = r16(ifd);
    if (ifd + 2 + 12ll * cnt > tn) return e;
    e.readable = true;
    // cv2 reads the entries in order and gives up on the segment at the first one whose data it cannot read.  An entry ahead of
    // the orientation is taken as read when it is in TIFF order (tag below 0x0112), of a known type, and its data is in the value
    // field or inside the segment.
    bool reached = true;
    for (int i = 0; i < cnt; ++i) {
        const int64_t q = ifd + 2 + 12ll * i;
        const int tag = r16(q);
        if (tag != 0x0112) {
            const int64_t bytes = type_bytes(r16(q + 2)) * r32(q + 4);
            reached = reached && tag < 0x0112 && type_bytes(r16(q + 2)) && (bytes <= 4 || r32(q + 8) + bytes <= tn);
            continue;
        }
        const bool shrt = r16(q + 2) == 3;
        if (e.tags++ == 0) e.value = shrt ? r16(q + 8) : 0;
        e.strict = e.strict && reached && shrt && r32(q + 4) == 1;
    }
    return e;
}

// A progressive parse (pn_jpeg_parse_progressive): the scans read so far and libjpeg's progression state.
struct Prog {
    pn_jpeg_scan scan[PN_JPEG_MAX_SCANS];
    pn_jpeg_huff huff[PN_JPEG_MAX_SCAN_HUFF];
    int n_scans, n_huff;
    int pool[2][4];          // huff[] index of a DHT slot's current definition, -1 before a scan uses it
    int coef_bits[3][64];    // jdphuff.c coef_bits: the last Al of each coefficient, -1 before its first scan
    bool latched[3];         // jdinput.c latch_quant_tables: a component's table is the one defined at its first scan
    void *out;               // the caller's table buffer, out_cap bytes
    int64_t out_cap, *out_bytes;
};

}  // namespace
}  // namespace pn

using namespace pn;

// One SOS of a progressive file (jdmarker.c get_sos, jdinput.c latch_quant_tables, jdphuff.c start_pass_phuff_decoder) at q, the
// byte after its length: records the scan, walks its entropy-coded data to the marker that ends it and leaves *p there.  Returns
// PN_JPEG_WHY_NONE, or why the file is the host's: anything libjpeg rejects or warns about.
template <class FrameWhy>
static int progressive_scan(const uint8_t *f, int64_t nbytes, pn_jpeg_desc *d, Prog &P, int64_t q, int ns, const int *comp_id,
                            const int *comp_h, const int *comp_v, const int *comp_tq, const bool hdef[2][4],
                            const uint8_t hbits[2][4][17], const uint8_t hvals[2][4][256], const bool *qdef,
                            const uint16_t qt[4][64], FrameWhy frame_why, int64_t *p) {
    const Reader R{f, nbytes};
    if (P.n_scans == 0) {                     // the frame: checks of the first scan, geometry of all components interleaved
        if (const int why = frame_why()) return why;
        const int all[3] = {0, 1, 2};
        if (!geometry(d, comp_h, comp_v, all, d->ncomp)) return PN_JPEG_WHY_SAMPLING;
    }
    if (P.n_scans == PN_JPEG_MAX_SCANS) return PN_JPEG_WHY_PROGRESSIVE;
    if (ns > d->ncomp) return PN_JPEG_WHY_UNKNOWN;
    pn_jpeg_scan &S = P.scan[P.n_scans];
    memset(&S, 0, sizeof(S));
    const int64_t o = q + 1 + 2 * ns;
    const int ss = R.u8(o), se = R.u8(o + 1), ah = R.u8(o + 2) >> 4, al = R.u8(o + 2) & 15;
    const bool dc = ss == 0;
    // JERR_BAD_PROGRESSION
    if ((dc ? se != 0 : ss > se || se > 63 || ns != 1) || (ah != 0 && al != ah - 1) || al > 13) return PN_JPEG_WHY_PROGRESSIVE;
    int blocks = 0;
    for (int s = 0; s < ns; ++s) {
        const int cid = R.u8(q + 1 + 2 * s), tdta = R.u8(q + 2 + 2 * s);
        int c = -1;
        for (int k = 0; k < d->ncomp; ++k)
            if (comp_id[k] == cid) c = k;
        for (int k = 0; k < s; ++k)
            if (S.comp[k] == c) c = -1;
        if (c < 0) return PN_JPEG_WHY_UNKNOWN;
        S.comp[s] = (uint8_t)c;
        blocks += comp_h[c] * comp_v[c];
        if (!P.latched[c]) {
            if (!qdef[comp_tq[c]]) return PN_JPEG_WHY_BAD_TABLE;
            for (int i = 0; i < 64; ++i) d->quant[c][i] = (int16_t)qt[comp_tq[c]][i];
            P.latched[c] = true;
        }
        if (!dc || ah == 0) {                 // DC refinement reads no table
            const int cls = dc ? 0 : 1, id = dc ? tdta >> 4 : tdta & 15;
            if (id > 3) return PN_JPEG_WHY_BAD_TABLE;
            if (!hdef[cls][id]) return PN_JPEG_WHY_NO_DHT;
            int &slot = P.pool[cls][id];
            if (slot < 0) {
                if (P.n_huff == PN_JPEG_MAX_SCAN_HUFF) return PN_JPEG_WHY_PROGRESSIVE;
                if (!derive(hbits[cls][id], hvals[cls][id], cls == 0, &P.huff[P.n_huff])) return PN_JPEG_WHY_BAD_TABLE;
                slot = P.n_huff++;
            }
            (dc ? S.dc[s] : S.ac[s]) = (uint8_t)slot;
        }
        // JWRN_BOGUS_PROGRESSION: an AC scan before the component's DC, or Ah other than the coefficient's last Al
        int *bits = P.coef_bits[c];
        if (!dc && bits[0] < 0) return PN_JPEG_WHY_PROGRESSIVE;
        for (int k = ss; k <= se; ++k) {
            if (ah != (bits[k] < 0 ? 0 : bits[k])) return PN_JPEG_WHY_PROGRESSIVE;
            bits[k] = al;
        }
    }
    if (ns > 1 && blocks > PN_JPEG_MAX_BLOCKS) return PN_JPEG_WHY_SAMPLING;
    S.ncomp = (uint8_t)ns;
    S.ss = (uint8_t)ss;
    S.se = (uint8_t)se;
    S.ah = (uint8_t)ah;
    S.al = (uint8_t)al;
    S.restart_interval = d->restart_interval;       // the DRI in force
    for (int t = 0; t < P.n_scans; ++t) {           // wave: one past the latest earlier scan on a shared (component, coefficient)
        const pn_jpeg_scan &T = P.scan[t];
        if (T.ss > se || ss > T.se) continue;
        bool shared = false;
        for (int a = 0; a < T.ncomp; ++a)
            for (int b = 0; b < ns; ++b) shared = shared || T.comp[a] == S.comp[b];
        if (shared && T.wave + 1 > S.wave) S.wave = T.wave + 1;
    }
    // the entropy-coded data runs to the first marker other than RSTn (0xFF 0x00 is a data byte, 0xFF fill bytes collapse)
    int64_t e = q + 4 + 2 * ns;
    for (;;) {
        const void *ff = e < nbytes ? memchr(f + e, 0xFF, (size_t)(nbytes - e)) : nullptr;
        if (!ff) return PN_JPEG_WHY_TRUNCATED;
        e = static_cast<const uint8_t *>(ff) - f;
        int64_t g = e + 1;
        while (g < nbytes && f[g] == 0xFF) ++g;
        if (g >= nbytes) return PN_JPEG_WHY_TRUNCATED;
        if (f[g] != 0 && (f[g] < 0xD0 || f[g] > 0xD7)) break;
        e = g + 1;
    }
    S.start = q + 4 + 2 * ns;
    S.end = e;
    ++P.n_scans;
    *p = e;
    return PN_JPEG_WHY_NONE;
}

// The EOI of a progressive file: a complete script becomes a PN_JPEG_SUPPORTED_PROGRESSIVE descriptor and its scan table.
static int finish_progressive(pn_jpeg_desc *d, Prog &P, int orientation) {
    // an incomplete script (a coefficient not refined to Al = 0) is decoded by libjpeg with block smoothing (jdcoefct.c)
    for (int c = 0; c < d->ncomp; ++c)
        for (int k = 0; k < 64; ++k)
            if (P.coef_bits[c][k] != 0) return host(d, PN_JPEG_WHY_PROGRESSIVE);
    const int64_t bytes = jpeg::scan_table_bytes(P.n_scans, P.n_huff);
    *P.out_bytes = bytes;
    if (bytes > P.out_cap) return host(d, PN_JPEG_WHY_PROGRESSIVE);
    pn_jpeg_scans h{P.n_scans, P.n_huff, 0, 0};
    for (int s = 0; s < P.n_scans; ++s) h.n_waves = P.scan[s].wave + 1 > h.n_waves ? P.scan[s].wave + 1 : h.n_waves;
    uint8_t *out = static_cast<uint8_t *>(P.out);
    memcpy(out, &h, sizeof(h));
    memcpy(out + sizeof(h), P.scan, sizeof(pn_jpeg_scan) * P.n_scans);
    memcpy(out + sizeof(h) + sizeof(pn_jpeg_scan) * P.n_scans, P.huff, sizeof(pn_jpeg_huff) * P.n_huff);
    const int64_t mcus = (int64_t)d->mcus_x * d->mcus_y;
    d->restart_interval = (int32_t)mcus;
    d->n_segments = 1;
    d->scan_offset = P.scan[0].start;
    d->kind = PN_JPEG_SUPPORTED_PROGRESSIVE;
    d->why = PN_JPEG_WHY_NONE;
    d->orientation = (uint8_t)orientation;
    return PN_OK;
}

// oriented: a file whose EXIF orientation o (2..8) is certain is PN_JPEG_SUPPORTED with desc->orientation = o (pn_jpeg_parse_oriented)
// pg: progressive files are decoded too (pn_jpeg_parse_progressive); null for the baseline parsers
static int parse(const uint8_t *file_host, int64_t nbytes, pn_jpeg_desc *d, bool oriented, Prog *pg) {
    memset(d, 0, sizeof(*d));
    d->file_bytes = nbytes;
    const Reader R{file_host, nbytes};
    if (R.u16(0) != 0xFFD8) return host(d, PN_JPEG_WHY_NOT_JPEG);

    uint8_t hbits[2][4][17] = {}, hvals[2][4][256] = {};
    bool hdef[2][4] = {};
    uint16_t qt[4][64] = {};
    bool qdef[4] = {};
    int comp_id[3] = {}, comp_h[3] = {}, comp_v[3] = {}, comp_tq[3] = {};
    bool sof = false, jfif = false, adobe = false, progressive = false;
    int adobe_transform = -1;
    // EXIF: any Exif segment that is unreadable or says other than 1 sends the file to the host (cv2 takes the first segment with
    // a readable orientation, looser than read_exif).  The oriented parse keeps a file whose Exif segments are all readable, whose
    // 0x0112 entries are single SHORTs that cv2 reaches, one per segment, and agree on one value o.
    bool exif_rotates = false, exif_certain = true;
    int exif_o = -1;                       // the value of the 0x0112 entries, -1 before the first
    // what sends the file to the host whatever its scans: an EXIF rotation the decode does not apply, RGB or unknown colour
    auto frame_why = [&]() -> int {
        const int orientation = exif_rotates ? exif_o : 0;
        if (exif_rotates && !(oriented && exif_certain && orientation >= 2 && orientation <= 8))
            return PN_JPEG_WHY_EXIF_ORIENTATION;
        if (d->ncomp == 3) {
            if (jfif) {
            } else if (adobe) {
                if (adobe_transform == 0) return PN_JPEG_WHY_RGB;
                if (adobe_transform != 1) return PN_JPEG_WHY_UNKNOWN;                     // libjpeg warns and assumes YCbCr
            } else if (comp_id[0] == 82 && comp_id[1] == 71 && comp_id[2] == 66) {
                return PN_JPEG_WHY_RGB;
            }
        }
        return PN_JPEG_WHY_NONE;
    };
    int64_t p = 2;
    for (;;) {
        if (R.u8(p) != 0xFF) return host(d, R.u8(p) < 0 ? PN_JPEG_WHY_TRUNCATED : PN_JPEG_WHY_UNKNOWN);   // extraneous bytes
        while (R.u8(p) == 0xFF) ++p;                                                                       // fill bytes
        const int m = R.u8(p++);
        if (m < 0) return host(d, PN_JPEG_WHY_TRUNCATED);
        if (m == 0xD9 && progressive && pg->n_scans) return finish_progressive(d, *pg, exif_rotates ? exif_o : 0);
        if (m == 0xD8 || m == 0xD9 || (m >= 0xD0 && m <= 0xD7) || m == 0x01) return host(d, PN_JPEG_WHY_UNKNOWN);
        const int len = R.u16(p);
        if (len < 0 || p + len > nbytes) return host(d, PN_JPEG_WHY_TRUNCATED);
        if (len < 2) return host(d, PN_JPEG_WHY_UNKNOWN);
        const int64_t q = p + 2, end = p + len;
        if (m == 0xC0 || m == 0xC1 || (pg && m == 0xC2)) {
            if (sof || len < 8) return host(d, PN_JPEG_WHY_UNKNOWN);
            sof = true;
            progressive = m == 0xC2;
            if (R.u8(q) != 8) return host(d, PN_JPEG_WHY_PRECISION);
            d->height = R.u16(q + 1);
            d->width = R.u16(q + 3);
            d->ncomp = R.u8(q + 5);
            if (d->height <= 0 || d->width <= 0 || d->height > 65500 || d->width > 65500) return host(d, PN_JPEG_WHY_UNKNOWN);
            if (d->ncomp != 1 && d->ncomp != 3) return host(d, PN_JPEG_WHY_COMPONENTS);
            if (len != 8 + 3 * d->ncomp) return host(d, PN_JPEG_WHY_UNKNOWN);
            for (int c = 0; c < d->ncomp; ++c) {
                comp_id[c] = R.u8(q + 6 + 3 * c);
                comp_h[c] = R.u8(q + 7 + 3 * c) >> 4;
                comp_v[c] = R.u8(q + 7 + 3 * c) & 15;
                comp_tq[c] = R.u8(q + 8 + 3 * c);
                if (comp_h[c] < 1 || comp_h[c] > 4 || comp_v[c] < 1 || comp_v[c] > 2 || comp_tq[c] > 3)
                    return host(d, PN_JPEG_WHY_SAMPLING);
            }
        } else if (m == 0xC2 || m == 0xC6) {
            return host(d, PN_JPEG_WHY_PROGRESSIVE);
        } else if (m == 0xC3 || m == 0xC7) {
            return host(d, PN_JPEG_WHY_LOSSLESS);
        } else if ((m >= 0xC9 && m <= 0xCB) || (m >= 0xCD && m <= 0xCF) || m == 0xCC) {
            return host(d, PN_JPEG_WHY_ARITHMETIC);
        } else if (m == 0xC5) {
            return host(d, PN_JPEG_WHY_UNKNOWN);                                          // differential
        } else if (m == 0xC4) {
            int64_t o = q;
            while (o < end) {
                const int tc = R.u8(o) >> 4, th = R.u8(o) & 15;
                if (tc > 1 || th > 3 || o + 17 > end) return host(d, PN_JPEG_WHY_BAD_TABLE);
                int count = 0;
                hbits[tc][th][0] = 0;
                for (int l = 1; l <= 16; ++l) count += (hbits[tc][th][l] = (uint8_t)R.u8(o + l));
                if (count > 256 || o + 17 + count > end) return host(d, PN_JPEG_WHY_BAD_TABLE);
                memset(hvals[tc][th], 0, 256);
                memcpy(hvals[tc][th], file_host + o + 17, count);
                hdef[tc][th] = true;
                if (pg) pg->pool[tc][th] = -1;           // the next scan that uses the slot derives the new definition
                o += 17 + count;
            }
        } else if (m == 0xDB) {
            int64_t o = q;
            while (o < end) {
                const int pq = R.u8(o) >> 4, tq = R.u8(o) & 15;
                if (pq > 1 || tq > 3 || o + 1 + 64 * (pq + 1) > end) return host(d, PN_JPEG_WHY_BAD_TABLE);
                for (int i = 0; i < 64; ++i)
                    qt[tq][jpeg::natural_order(i)] = (uint16_t)(pq ? R.u16(o + 1 + 2 * i) : R.u8(o + 1 + i));
                qdef[tq] = true;
                o += 1 + 64 * (pq + 1);
            }
        } else if (m == 0xDD) {
            if (len != 4) return host(d, PN_JPEG_WHY_UNKNOWN);
            d->restart_interval = R.u16(q);
        } else if (m == 0xE0) {
            if (len - 2 >= 14 && !memcmp(file_host + q, "JFIF\0", 5)) jfif = true;
        } else if (m == 0xE1) {
            if (len - 2 >= 6 && !memcmp(file_host + q, "Exif\0\0", 6)) {
                if (pg && pg->n_scans) return host(d, PN_JPEG_WHY_EXIF_ORIENTATION);   // past the headers cv2 reads it from
                const Exif e = read_exif(file_host + q, len - 2);
                exif_rotates = exif_rotates || !e.readable || e.value != 1;
                exif_certain = exif_certain && e.readable && e.strict && e.tags <= 1;
                if (e.tags && exif_o >= 0 && exif_o != e.value) exif_certain = false;
                if (e.tags) exif_o = e.value;
            }
        } else if (m == 0xEE) {
            if (len - 2 >= 12 && !memcmp(file_host + q, "Adobe", 5)) {
                adobe = true;
                adobe_transform = R.u8(q + 11);
            }
        } else if ((m >= 0xE2 && m <= 0xEF) || m == 0xFE) {
            // other application data and comments: skipped
        } else if (m == 0xDA) {
            if (!sof) return host(d, PN_JPEG_WHY_UNKNOWN);
            const int ns = R.u8(q);
            if (ns < 1 || ns > 4 || len != 6 + 2 * ns) return host(d, PN_JPEG_WHY_UNKNOWN);
            if (progressive) {
                const int why = progressive_scan(file_host, nbytes, d, *pg, q, ns, comp_id, comp_h, comp_v, comp_tq, hdef, hbits,
                                                 hvals, qdef, qt, frame_why, &p);
                if (why != PN_JPEG_WHY_NONE) return host(d, why);
                continue;
            }
            if (ns != d->ncomp) return host(d, PN_JPEG_WHY_MULTI_SCAN);
            if (R.u8(q + 1 + 2 * ns) != 0 || R.u8(q + 2 + 2 * ns) != 63 || R.u8(q + 3 + 2 * ns) != 0)
                return host(d, PN_JPEG_WHY_UNKNOWN);                                      // Ss, Se, Ah/Al of a sequential scan
            const int orientation = exif_rotates ? exif_o : 0;
            if (const int why = frame_why()) return host(d, why);
            // huffman slots: up to four distinct (class, id) pairs
            int slot_key[4], nslots = 0;
            int order[3];
            for (int s = 0; s < ns; ++s) {
                const int cid = R.u8(q + 1 + 2 * s), tdta = R.u8(q + 2 + 2 * s);
                int c = -1;
                for (int k = 0; k < d->ncomp; ++k)
                    if (comp_id[k] == cid) c = k;
                for (int k = 0; k < s; ++k)
                    if (order[k] == c) c = -1;
                if (c < 0) return host(d, PN_JPEG_WHY_UNKNOWN);
                order[s] = c;
                const int td = tdta >> 4, ta = tdta & 15;
                if (td > 3 || ta > 3) return host(d, PN_JPEG_WHY_BAD_TABLE);
                if (!hdef[0][td] || !hdef[1][ta]) return host(d, PN_JPEG_WHY_NO_DHT);
                if (!qdef[comp_tq[c]]) return host(d, PN_JPEG_WHY_BAD_TABLE);
                for (int cls = 0; cls < 2; ++cls) {
                    const int key = cls * 4 + (cls ? ta : td);
                    int sl = -1;
                    for (int k = 0; k < nslots; ++k)
                        if (slot_key[k] == key) sl = k;
                    if (sl < 0) {
                        if (nslots == 4) return host(d, PN_JPEG_WHY_UNKNOWN);
                        sl = nslots;
                        slot_key[nslots++] = key;
                        if (!derive(hbits[cls][key & 3], hvals[cls][key & 3], cls == 0, &d->huff[sl]))
                            return host(d, PN_JPEG_WHY_BAD_TABLE);
                    }
                    (cls ? d->comp[c].ac : d->comp[c].dc) = sl;
                }
                for (int i = 0; i < 64; ++i) d->quant[c][i] = (int16_t)qt[comp_tq[c]][i];
            }
            if (!geometry(d, comp_h, comp_v, order, ns)) return host(d, PN_JPEG_WHY_SAMPLING);
            const int64_t mcus = (int64_t)d->mcus_x * d->mcus_y;
            if (d->restart_interval <= 0 || d->restart_interval > mcus) d->restart_interval = (int32_t)mcus;
            d->n_segments = (int32_t)((mcus + d->restart_interval - 1) / d->restart_interval);
            d->scan_offset = end;
            // the scan must be followed by a marker: a file cut short (no EOI after the scan) is cv2's to patch up
            bool eoi = false;
            for (int64_t o = nbytes - 2; o >= end && !eoi; --o) eoi = file_host[o] == 0xFF && file_host[o + 1] == 0xD9;
            if (!eoi) return host(d, PN_JPEG_WHY_TRUNCATED);
            d->kind = PN_JPEG_SUPPORTED;
            d->why = PN_JPEG_WHY_NONE;
            d->orientation = (uint8_t)orientation;
            return PN_OK;
        } else {
            return host(d, PN_JPEG_WHY_UNKNOWN);                                          // DNL, DHP, EXP, JPG, ...
        }
        p = end;
    }
}

extern "C" int pn_jpeg_parse(const uint8_t *file_host, int64_t nbytes, pn_jpeg_desc *d) {
    PN_CHECK_ARG(file_host && d && nbytes >= 0, "pn_jpeg_parse: null pointer or negative size");
    return parse(file_host, nbytes, d, false, nullptr);
}

extern "C" int pn_jpeg_parse_oriented(const uint8_t *file_host, int64_t nbytes, pn_jpeg_desc *d) {
    PN_CHECK_ARG(file_host && d && nbytes >= 0, "pn_jpeg_parse_oriented: null pointer or negative size");
    return parse(file_host, nbytes, d, true, nullptr);
}

extern "C" int pn_jpeg_parse_progressive(const uint8_t *file_host, int64_t nbytes, int oriented, pn_jpeg_desc *d, void *scans_host,
                                         int64_t scans_cap, int64_t *scans_bytes) {
    PN_CHECK_ARG(file_host && d && scans_bytes && nbytes >= 0 && scans_cap >= 0 && (scans_host || !scans_cap),
                 "pn_jpeg_parse_progressive: null pointer or negative size");
    Prog pg;
    pg.n_scans = pg.n_huff = 0;
    memset(pg.pool, 0xFF, sizeof(pg.pool));
    memset(pg.coef_bits, 0xFF, sizeof(pg.coef_bits));
    memset(pg.latched, 0, sizeof(pg.latched));
    pg.out = scans_host;
    pg.out_cap = scans_cap;
    pg.out_bytes = scans_bytes;
    *scans_bytes = 0;
    return parse(file_host, nbytes, d, oriented != 0, &pg);
}
