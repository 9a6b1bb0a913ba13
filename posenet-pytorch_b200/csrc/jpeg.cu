// pn_jpeg_decode: baseline JPEG files -> uint8 BGR frames on the device, bit-exact with cv2.imdecode (arithmetic: jpeg_decode.cuh).
//
// One call decodes a batch in eleven launches whose geometry depends only on the arguments (so the call can be captured in a graph):
//   plan      validate every descriptor (a warp per image) and size its share of the workspace
//   layout    exclusive prefix sums of the shares (one CTA)
//   destuff   one CTA per image: drop 0xFF00 stuffing, find the restart markers and the end of the scan, cut every restart
//             interval (segment) into subsequences of SUB_BITS bits
//   spec      every subsequence (but a segment's last) decodes speculatively from its first bit as if block 0 of an MCU began
//             there, to the first codeword boundary at or past its end: exit state E1 (bit position, block in MCU, zig-zag index)
//   merge     every such subsequence follows its speculative path on until the path's state at the end of a later subsequence j
//             equals E1[j] (Huffman codes resynchronise, after which the two paths are one): the merge point m and the blocks
//             begun on the way -- the intra-sequence synchronisation of Weissenberger & Schmidt
//   walk      one warp per segment chases the merge points from subsequence 0, whose start is exact: the true path is path 0
//             up to m[0], then path m[0], ...  Every chain element gets its true exit state and block count
//   write     every subsequence decodes from its true entry and stores the blocks that begin in it (DC as a difference)
//   progressive  one warp per progressive image (pn_jpeg_parse_progressive's kind 2): its waves in order, the lanes decoding the
//             (scan, restart segment) pairs of a wave serially from the raw file bytes into the zeroed coefficient array
//             (jpeg_progressive.cuh).  The stages from destuff to write and dc have nothing to do for such an image
//   dc        one warp per segment: per-component prefix sums of the DC differences (reset at every restart marker)
//   idct      eight threads per block, into per-component sample planes: jpeg_idct_islow, or at 1/2, 1/4, 1/8 (scale_denom,
//             cv2's IMREAD_REDUCED_COLOR_*) the component's scaled IDCT (jidctred.c), ssize x ssize samples per block
//   color     upsampling + YCbCr -> BGR, one thread per output pixel, straight into the frame's row (ceil(h / d) x ceil(w / d)),
//             with the descriptor's EXIF orientation applied: flips map each output pixel to its source pixel, transposes stage
//             32 x 32 tiles through shared memory so that both the planes and the frame are walked along their rows
// Everything up to dc is independent of the scale and the orientation.  The workspace is sized for files of scale_denom * max_h x
// scale_denom * max_w in either order (a file whose reduced, oriented frame fits max_h x max_w is at most that large).
// (Weissenberger & Schmidt, "Massively Parallel Huffman Decoding on GPUs", ICPP 2018, for the self-synchronisation.)
#include "common.cuh"
#include "jpeg_decode.cuh"
#include "jpeg_progressive.cuh"

namespace pn {
namespace {

using namespace jpeg;

// Subsequence length.  A speculative decode meets the true path at the end of its own subsequence at 62-67 % of the boundaries of
// smooth q90 4:2:0 scans and 19-25 % of noisy ones (start guessed as block 0 of an MCU); the merge continuation covers the rest,
// so the serial depth is the synchronisation distance of the data (a few thousand bits smooth, ~30 kbit noisy q95 4:4:4), not
// SUB_BITS.  Shorter subsequences mean more threads and more boundaries to chase.
constexpr int SUB_BITS = 1024;
constexpr int MERGE_LIMIT = 64;  // subsequences a path is followed before the walk takes over serially
constexpr int THREADS = 256;

struct Totals {
    long long nseg, nsub, nblk;
};
struct ImgWs {
    int status;
    uint32_t ds_len;
    int seg_base, nseg, sub_base, sub_cap, nsub, pad;
    long long blk_base, nblk;
    long long plane_base[3];
};
struct SegWs {
    uint32_t start, end;       // byte range of the de-stuffed segment, from the image's de-stuffed base
    int sub_first, nsub;       // subsequences: slots sub_base + sub_first ..
};
struct SubInfo {
    int img, seg, k, nk;       // seg: global segment index
};

struct Layout {
    size_t totals, img, seg, sub, e1, ech, m, flag, c1, c2, bch, coef, planes, ds, bytes;
    long long nseg_cap, nsub_cap, nblk_cap;
};

size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

Layout layout(int n_img, int64_t arena, int max_h, int max_w) {
    Layout L;
    const long long bx = (max_w + 7) / 8, by = (max_h + 7) / 8;
    L.nseg_cap = (long long)n_img * bx * by;
    L.nsub_cap = L.nseg_cap + arena * 8 / SUB_BITS + n_img;
    // MCU padding of sampling factors up to 4 x 2, for a file of max_h x max_w or (transposed orientations) max_w x max_h
    L.nblk_cap = (long long)n_img * 3 * ((bx + 3) * (by + 1) > (by + 3) * (bx + 1) ? (bx + 3) * (by + 1) : (by + 3) * (bx + 1));
    size_t o = 0;
    auto take = [&](size_t bytes) { const size_t at = o; o = align256(o + bytes); return at; };
    L.totals = take(sizeof(Totals));
    L.img = take(sizeof(ImgWs) * n_img);
    L.seg = take(sizeof(SegWs) * L.nseg_cap);
    L.sub = take(sizeof(SubInfo) * L.nsub_cap);
    L.e1 = take(8 * L.nsub_cap);
    L.ech = take(8 * L.nsub_cap);
    L.m = take(4 * L.nsub_cap);
    L.flag = take(4 * L.nsub_cap);
    L.c1 = take(4 * L.nsub_cap);
    L.c2 = take(4 * L.nsub_cap);
    L.bch = take(4 * L.nsub_cap);
    L.coef = take(128 * L.nblk_cap);
    L.planes = take(64 * L.nblk_cap);
    L.ds = take(arena + 16);
    L.bytes = o;
    return L;
}

struct Ws {
    Totals *totals;
    ImgWs *img;
    SegWs *seg;
    SubInfo *sub;
    uint64_t *e1, *ech;          // speculative exits; true states the walk recorded serially (flag 2)
    int *m, *flag;                // merge points; chain marks (0 off the chain, 1 true state = e1, 2 true state = ech)
    uint32_t *c1, *c2, *bch;      // blocks begun: speculative decode, merge continuation, true path up to a chain element
    int16_t *coef;
    uint8_t *planes, *ds;
    long long nseg_cap, nsub_cap, nblk_cap;
};

struct Args {
    const uint8_t *files;
    int64_t arena;
    const pn_jpeg_desc *descs;
    int n_img, max_h, max_w, denom;    // max_h x max_w: the largest OUTPUT frame (at 1 / denom)
    uint8_t *frames;
    int64_t stride;
    int *frame_hw, *status;
};

__device__ __forceinline__ void fail(ImgWs &w, int code) { atomicMin(&w.status, code); }

__device__ __forceinline__ long long seg_blocks(const pn_jpeg_desc &d, int s) {
    const long long mcus = (long long)d.mcus_x * d.mcus_y;
    const long long first = (long long)s * d.restart_interval;
    const long long n = mcus - first < d.restart_interval ? mcus - first : d.restart_interval;
    return n * d.blocks_per_mcu;
}

__device__ __forceinline__ BitSrc seg_src(const Ws &ws, const pn_jpeg_desc &d, const SegWs &sg) {
    return BitSrc{ws.ds + d.file_offset + sg.start, sg.end - sg.start};
}

// A progressive descriptor's scan table (the warp of plan_kernel; the descriptor's own fields are checked there): inside the arena
// and 8-byte aligned, every scan a legal one over the frame's components with its bytes inside the file and its tables in the
// table, DC tables with symbols <= 15, and no two scans of one wave on a shared (component, coefficient) -- nor a scan in a wave
// at or before one it depends on.
__device__ bool scan_table_ok(const Args &a, const pn_jpeg_desc &d, int lane) {
    const int64_t t = scan_table_offset(d);
    const bool head_ok = d.file_offset >= 0 && d.file_bytes > 0 && t + (int64_t)sizeof(pn_jpeg_scans) <= a.arena &&
                         ((uintptr_t)(a.files + t) & 7) == 0;
    if (!__all_sync(0xffffffffu, head_ok)) return false;
    const uint8_t *tab = a.files + t;
    const pn_jpeg_scans h = *reinterpret_cast<const pn_jpeg_scans *>(tab);
    if (h.n_scans < 1 || h.n_scans > PN_JPEG_MAX_SCANS || h.n_huff < 0 || h.n_huff > PN_JPEG_MAX_SCAN_HUFF || h.n_waves < 1 ||
        h.n_waves > h.n_scans || t + scan_table_bytes(h.n_scans, h.n_huff) > a.arena)
        return false;
    const pn_jpeg_scan *sc = table_scans(tab);
    const pn_jpeg_huff *huff = table_huff(tab);
    bool ok = true;
    for (int s = lane; s < h.n_scans; s += 32) {
        const pn_jpeg_scan S = sc[s];
        const bool dc = S.ss == 0;
        bool g = S.ncomp >= 1 && S.ncomp <= d.ncomp && S.se <= 63 && S.ss <= S.se && (dc ? S.se == 0 : S.ncomp == 1) &&
                 S.al <= 13 && S.ah <= 13 && S.wave >= 0 && S.wave < h.n_waves && S.restart_interval >= 0 && S.start >= 0 &&
                 S.start <= S.end && S.end <= d.file_bytes;
        int blocks = 0;
        for (int i = 0; g && i < S.ncomp; ++i) {
            const int c = S.comp[i];
            g = c < d.ncomp;
            for (int j = 0; g && j < i; ++j) g = S.comp[j] != c;
            if (!g) break;
            blocks += d.comp[c].h * d.comp[c].v;
            if (dc && S.ah == 0) {
                g = S.dc[i] < h.n_huff;
                for (int e = 0; g && e < 256; ++e) g = (huff[S.dc[i]].lookup[e] & 0xFF) <= 15 && huff[S.dc[i]].huffval[e] <= 15;
            }
            if (!dc) g = g && S.ac[i] < h.n_huff;
        }
        g = g && blocks <= PN_JPEG_MAX_BLOCKS;
        for (int u = 0; g && u < s; ++u) {
            const pn_jpeg_scan &T = sc[u];
            bool shared = false;
            for (int x = 0; x < T.ncomp && x < 3; ++x)
                for (int y = 0; y < S.ncomp; ++y) shared = shared || T.comp[x] == S.comp[y];
            g = !(shared && T.ss <= S.se && S.ss <= T.se) || T.wave < S.wave;
        }
        ok = ok && g;
    }
    return __all_sync(0xffffffffu, ok);
}

// ---- plan: one warp per image validates its descriptor and sizes its share of the workspace ----------------------------------
__global__ void __launch_bounds__(32) plan_kernel(Args a, Ws ws) {
    const int lane = threadIdx.x, i = blockIdx.x;
        const pn_jpeg_desc &d = a.descs[i];
        const bool prog = d.kind == PN_JPEG_SUPPORTED_PROGRESSIVE;
        bool ok = d.kind == PN_JPEG_SUPPORTED || prog;
        const bool skipped = !ok;
        const long long rh = ((long long)d.height + a.denom - 1) / a.denom, rw = ((long long)d.width + a.denom - 1) / a.denom;
        const bool tr = orient_transposes(d.orientation);          // the oriented frame is rw x rh
        ok = ok && d.file_offset >= 0 && d.file_bytes > 0 && d.file_offset + d.file_bytes <= a.arena && d.scan_offset >= 0 &&
             d.scan_offset < d.file_bytes && d.height >= 1 && d.width >= 1 && d.orientation <= 8 && (tr ? rw : rh) <= a.max_h &&
             (tr ? rh : rw) <= a.max_w &&
             (d.ncomp == 1 || d.ncomp == 3) && d.blocks_per_mcu >= 1 && d.blocks_per_mcu <= PN_JPEG_MAX_BLOCKS &&
             d.mcus_x >= 1 && d.mcus_y >= 1 && d.restart_interval >= 1;
        const long long mcus = ok ? (long long)d.mcus_x * d.mcus_y : 0;
        ok = ok && d.n_segments == (mcus + d.restart_interval - 1) / d.restart_interval;
        long long planes = 0;
        for (int c = 0; ok && c < d.ncomp; ++c) {
            const pn_jpeg_comp &k = d.comp[c];
            ok = k.h >= 1 && k.h <= 4 && k.v >= 1 && k.v <= 4 && k.hr >= 1 && k.vr >= 1 && k.dc >= 0 && k.dc < 4 && k.ac >= 0 &&
                 k.ac < 4 && k.bw == d.mcus_x * k.h && k.bh == d.mcus_y * k.v && k.dw >= 1 && k.dh >= 1 && k.dw <= 8 * k.bw &&
                 k.dh <= 8 * k.bh && (d.width - 1) / k.hr < k.dw && (d.height - 1) / k.vr < k.dh;
            planes += (long long)k.bw * k.bh;
        }
        for (int b = 0; ok && b < d.blocks_per_mcu; ++b) {
            const int c = d.mcu_comp[b];
            ok = c < d.ncomp && d.mcu_bx[b] < d.comp[c].h && d.mcu_by[b] < d.comp[c].v;
        }
        ok = ok && planes == mcus * d.blocks_per_mcu;
        Scaled g;                              // the reduced planes and the upsampler's reads stay inside the blocks
        ok = ok && scaled_geometry(d, a.denom, &g);
        for (int c = 0; ok && c < d.ncomp; ++c) {
            const pn_jpeg_comp &k = d.comp[c];
            const CompScale &s = g.comp[c];
            ok = s.dw >= 1 && s.dh >= 1 && s.dw <= s.ssize * k.bw && s.dh <= s.ssize * k.bh && (g.w - 1) / s.hr < s.dw &&
                 (g.h - 1) / s.vr < s.dh;
        }
        // DC symbols are extra-bit counts: at most 15 (what jpeg_make_d_derived_tbl enforces)
        bool tables_ok = true;
        for (int c = 0; ok && !prog && c < d.ncomp; ++c) {
            const pn_jpeg_huff &t = d.huff[d.comp[c].dc];
            for (int e = lane; e < 256; e += 32) tables_ok &= (t.lookup[e] & 0xFF) <= 15 && t.huffval[e] <= 15;
        }
        if (prog) ok = ok && canonical_mcu(d) && scan_table_ok(a, d, lane);
        ok = ok && __all_sync(0xffffffffu, tables_ok);
        if (lane == 0) {
            ImgWs &w = ws.img[i];
            w.status = skipped ? PN_JPEG_SKIPPED : ok ? PN_JPEG_OK : PN_JPEG_ERR_DESC;
            w.ds_len = 0;
            w.nseg = ok && !prog ? d.n_segments : 0;
            w.sub_cap = ok && !prog ? (int)(d.n_segments + d.file_bytes * 8 / SUB_BITS) : 0;
            w.nsub = 0;
            w.nblk = ok ? mcus * d.blocks_per_mcu : 0;
            long long pb = 0;                  // plane offsets within the image's share; layout_kernel adds its base
            for (int c = 0; c < 3; ++c) {
                w.plane_base[c] = pb;
                if (ok && c < d.ncomp) pb += 64ll * d.comp[c].bw * d.comp[c].bh;
            }
        }
}

// ---- layout: exclusive prefix sums of the images' shares (one CTA); an image past a capacity is a descriptor error ------------
template <typename T>
__device__ T block_exclusive_scan(T v, T *total, T *sm);

__global__ void __launch_bounds__(THREADS, 1) layout_kernel(Args a, Ws ws) {
    __shared__ long long sm[THREADS / 32 + 1];
    __shared__ unsigned long long s_end[3];
    if (threadIdx.x < 3) s_end[threadIdx.x] = 0;
    long long carry[3] = {0, 0, 0};
    for (int i0 = 0; i0 < a.n_img; i0 += THREADS) {
        const int i = i0 + threadIdx.x;
        ImgWs *w = i < a.n_img ? &ws.img[i] : nullptr;
        const bool ok = w && w->status == PN_JPEG_OK;
        const long long own[3] = {ok ? w->nseg : 0, ok ? w->sub_cap : 0, ok ? w->nblk : 0};
        const long long cap[3] = {ws.nseg_cap, ws.nsub_cap, ws.nblk_cap};
        long long base[3];
        bool fits = true;
        for (int q = 0; q < 3; ++q) {
            long long tot;
            base[q] = block_exclusive_scan<long long>(own[q], &tot, sm) + carry[q];
            carry[q] += tot;
            fits = fits && base[q] + own[q] <= cap[q];
        }
        if (w) {
            w->seg_base = (int)base[0];
            w->sub_base = (int)base[1];
            w->blk_base = base[2];
            for (int c = 0; c < 3; ++c) w->plane_base[c] += base[2] * 64;
            if (ok && !fits) {
                w->status = PN_JPEG_ERR_DESC;
            } else if (ok) {
                for (int q = 0; q < 3; ++q) atomicMax(&s_end[q], (unsigned long long)(base[q] + own[q]));
            }
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) *ws.totals = Totals{(long long)s_end[0], (long long)s_end[1], (long long)s_end[2]};
}

// ---- destuff: one CTA per image ----------------------------------------------------------------------------------------------------
template <typename T>
__device__ T block_exclusive_scan(T v, T *total, T *sm) {   // sm: THREADS / 32 + 1 entries
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    T x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const T y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) sm[warp] = x;
    __syncthreads();
    if (threadIdx.x == 0) {
        T run = 0;
        for (int k = 0; k < THREADS / 32; ++k) {
            const T t = sm[k];
            sm[k] = run;
            run += t;
        }
        sm[THREADS / 32] = run;
    }
    __syncthreads();
    const T r = sm[warp] + x - v;
    *total = sm[THREADS / 32];
    __syncthreads();
    return r;
}

constexpr int DS_PER_THREAD = 8;

__global__ void __launch_bounds__(THREADS, 1) destuff_kernel(Args a, Ws ws) {
    const int i = blockIdx.x;
    ImgWs &w = ws.img[i];
    if (w.status != PN_JPEG_OK || a.descs[i].kind != PN_JPEG_SUPPORTED) return;
    const pn_jpeg_desc &d = a.descs[i];
    const uint8_t *f = a.files + d.file_offset;
    const long long n = d.file_bytes, p0 = d.scan_offset;
    uint8_t *out = ws.ds + d.file_offset;
    SegWs *seg = ws.seg + w.seg_base;
    __shared__ long long s_end;
    __shared__ uint32_t s_nout, s_nrst;
    __shared__ int s_bad;
    __shared__ uint32_t sm_u[THREADS / 32 + 1];
    __shared__ int sm_i[THREADS / 32 + 1];
    if (threadIdx.x == 0) {
        s_end = LLONG_MAX;
        s_nout = 0;
        s_nrst = 0;
        s_bad = 0;
    }
    __syncthreads();
    for (long long chunk = p0; chunk < n; chunk += THREADS * DS_PER_THREAD) {
        const long long q0 = chunk + (long long)threadIdx.x * DS_PER_THREAD;
        uint8_t kind[DS_PER_THREAD];
        long long my_end = LLONG_MAX;
#pragma unroll
        for (int j = 0; j < DS_PER_THREAD; ++j) {
            const long long q = q0 + j;
            if (q >= n) {
                kind[j] = BYTE_DROP;
                continue;
            }
            const int prev = q > p0 ? f[q - 1] : -1, next = q + 1 < n ? f[q + 1] : -1;
            kind[j] = (uint8_t)classify_byte(prev, f[q], next);
            if (kind[j] == BYTE_END && q < my_end) my_end = q;
        }
        if (my_end != LLONG_MAX) atomicMin((unsigned long long *)&s_end, (unsigned long long)my_end);
        __syncthreads();
        const long long end = s_end;
        uint32_t nd = 0;
        int nr = 0;
#pragma unroll
        for (int j = 0; j < DS_PER_THREAD; ++j) {
            if (q0 + j >= end) kind[j] = BYTE_DROP;
            nd += kind[j] == BYTE_DATA;
            nr += kind[j] == BYTE_RST;
        }
        uint32_t tot_d;
        int tot_r;
        uint32_t od = block_exclusive_scan<uint32_t>(nd, &tot_d, sm_u) + s_nout;
        int orr = block_exclusive_scan<int>(nr, &tot_r, sm_i) + (int)s_nrst;
#pragma unroll
        for (int j = 0; j < DS_PER_THREAD; ++j) {
            if (kind[j] == BYTE_DATA) {
                out[od++] = f[q0 + j];
            } else if (kind[j] == BYTE_RST) {
                if (f[q0 + j + 1] - 0xD0 != (orr & 7)) s_bad = 1;
                if (orr + 1 < w.nseg) seg[orr + 1].start = od;
                ++orr;
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            s_nout += tot_d;
            s_nrst += (uint32_t)tot_r;
        }
        __syncthreads();
        if (end != LLONG_MAX) break;
    }
    const int nseg = w.nseg;
    int status = PN_JPEG_OK;
    if (s_end == LLONG_MAX) status = PN_JPEG_ERR_NO_END;
    else if (s_bad || (int)s_nrst != nseg - 1) status = PN_JPEG_ERR_RESTART;
    const uint32_t ds_len = s_nout;
    if (status == PN_JPEG_OK) {
        if (threadIdx.x == 0) seg[0].start = 0;
        __syncthreads();
        // segment ends and subsequence counts, prefix-summed in chunks of THREADS segments
        __shared__ int s_run;
        if (threadIdx.x == 0) s_run = 0;
        __syncthreads();
        for (int s0 = 0; s0 < nseg; s0 += THREADS) {
            const int s = s0 + threadIdx.x;
            int nk = 0;
            if (s < nseg) {
                const uint32_t st = seg[s].start, en = s + 1 < nseg ? seg[s + 1].start : ds_len;
                if (en <= st) s_bad = 1;
                const uint32_t bits = (en - st) * 8u;
                nk = bits / SUB_BITS > 1 ? (int)(bits / SUB_BITS) : 1;
                seg[s].end = en;
                seg[s].nsub = nk;
            }
            int tot;
            const int off = block_exclusive_scan<int>(nk, &tot, sm_i) + s_run;
            if (s < nseg) seg[s].sub_first = off;
            __syncthreads();
            if (threadIdx.x == 0) s_run += tot;
            __syncthreads();
        }
        if (s_bad) status = PN_JPEG_ERR_LENGTH;
        const int nsub = s_run;
        if (status == PN_JPEG_OK && nsub > w.sub_cap) status = PN_JPEG_ERR_LENGTH;   // cannot happen: sum of floors <= floor of sum
        if (status == PN_JPEG_OK) {
            for (int s = threadIdx.x; s < nseg; s += THREADS)
                for (int k = 0; k < seg[s].nsub; ++k)
                    ws.sub[w.sub_base + seg[s].sub_first + k] = SubInfo{i, w.seg_base + s, k, seg[s].nsub};
            for (int j = nsub + threadIdx.x; j < w.sub_cap; j += THREADS) ws.sub[w.sub_base + j].img = -1;
            if (threadIdx.x == 0) {
                w.nsub = nsub;
                w.ds_len = ds_len;
            }
            return;
        }
    }
    for (int j = threadIdx.x; j < w.sub_cap; j += THREADS) ws.sub[w.sub_base + j].img = -1;
    if (threadIdx.x == 0) fail(w, status);
}

// ---- speculative decodes ---------------------------------------------------------------------------------------------------------
// spec: every subsequence but a segment's last decodes from its first bit as if a block 0 began there: exit E1, blocks c1.
__global__ void __launch_bounds__(THREADS) spec_kernel(Args a, Ws ws) {
    const long long total = ws.totals->nsub;
    for (long long j = blockIdx.x * (long long)THREADS + threadIdx.x; j < total; j += (long long)gridDim.x * THREADS) {
        const SubInfo info = ws.sub[j];
        if (info.img < 0 || info.k == info.nk - 1 || ws.img[info.img].status != PN_JPEG_OK) continue;
        const pn_jpeg_desc &d = a.descs[info.img];
        const BitSrc src = seg_src(ws, d, ws.seg[info.seg]);
        State s{(uint32_t)info.k * SUB_BITS, 0, 0};
        uint32_t blocks = 0;
        const bool ok = advance(d, src, s, (uint32_t)(info.k + 1) * SUB_BITS, &blocks);
        ws.e1[j] = ok ? pack(s) : kBadState;
        ws.c1[j] = blocks;
    }
}

// merge: every such subsequence follows its speculative path on from E1 until it meets a later subsequence's E1 (merge_point):
// the index m of that subsequence (or MERGE_TAIL / MERGE_NONE) and the blocks begun on the way, c2.
__global__ void __launch_bounds__(THREADS) merge_kernel(Args a, Ws ws) {
    const long long total = ws.totals->nsub;
    for (long long j = blockIdx.x * (long long)THREADS + threadIdx.x; j < total; j += (long long)gridDim.x * THREADS) {
        const SubInfo info = ws.sub[j];
        if (info.img < 0 || info.k == info.nk - 1 || ws.img[info.img].status != PN_JPEG_OK) continue;
        const uint64_t e = ws.e1[j];
        uint32_t blocks = 0;
        int m = MERGE_NONE;
        if (e != kBadState) {
            const pn_jpeg_desc &d = a.descs[info.img];
            const uint64_t *e1 = ws.e1 + (j - info.k);
            m = merge_point(d, seg_src(ws, d, ws.seg[info.seg]), unpack(e), info.k, info.nk, SUB_BITS, MERGE_LIMIT,
                            [e1](int jj) { return e1[jj]; }, &blocks);
        }
        ws.m[j] = m;
        ws.c2[j] = blocks;
    }
}

// ---- walk: one warp per segment follows the chain of merge points ----------------------------------------------------------------
// The true path leaves subsequence 0 in state E1[0]; it is path 0, which joins path m[0] at the end of m[0], and so on.  The
// warp marks the chain (flag 1: the true state at the end of k is E1[k]) with the blocks begun up to there (bch), chasing m[] in
// shared-memory windows.  A chain element whose path met no later E1 within MERGE_LIMIT subsequences (rare; a corrupt scan) is
// followed by lane 0 alone, one subsequence at a time, recording each state (flag 2, ech) until it meets an E1 again.
constexpr int WALK_WIN = 256;
__global__ void __launch_bounds__(THREADS, 1) walk_kernel(Args a, Ws ws) {
    __shared__ int sm_m[THREADS / 32][WALK_WIN];
    __shared__ uint32_t sm_c[THREADS / 32][WALK_WIN];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const long long warps = (long long)gridDim.x * (THREADS / 32);
    const long long total = ws.totals->nseg;
    for (long long sgi = blockIdx.x * (long long)(THREADS / 32) + wid; sgi < total; sgi += warps) {
        const SegWs sg = ws.seg[sgi];
        int lo = 0, hi = a.n_img - 1;          // the image: last one whose segments start at or before sgi
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (ws.img[mid].seg_base <= sgi) lo = mid; else hi = mid - 1;
        }
        ImgWs &w = ws.img[lo];
        if (w.status != PN_JPEG_OK) continue;
        const long long j0 = w.sub_base + sg.sub_first;
        const int nk = sg.nsub;
        for (int r = lane; r < nk; r += 32) ws.flag[j0 + r] = 0;
        __syncwarp();
        if (nk == 1) continue;
        if (ws.e1[j0] == kBadState) {
            if (lane == 0) fail(w, PN_JPEG_ERR_CODE);
            continue;
        }
        const pn_jpeg_desc &d = a.descs[lo];
        int c = 0;
        uint32_t cum = ws.c1[j0];
        if (lane == 0) {
            ws.flag[j0] = 1;
            ws.bch[j0] = cum;
        }
        int status = 0;                        // 0 chase on, 1 chain complete, 2 follow serially, 3 bad code
        while (status == 0 || status == 2) {
            if (status == 0) {
                for (int i = lane; i < WALK_WIN; i += 32) {
                    const int kk = c + i;
                    sm_m[wid][i] = kk < nk - 1 ? ws.m[j0 + kk] : MERGE_TAIL;
                    sm_c[wid][i] = kk < nk - 1 ? ws.c2[j0 + kk] : 0u;
                }
                __syncwarp();
                if (lane == 0) {
                    const int w0 = c;
                    for (;;) {
                        const int m = sm_m[wid][c - w0];
                        if (m == MERGE_TAIL) { status = 1; break; }
                        if (m == MERGE_NONE) { status = 2; break; }
                        cum += sm_c[wid][c - w0];
                        c = m;
                        ws.flag[j0 + c] = 1;
                        ws.bch[j0 + c] = cum;
                        if (c - w0 >= WALK_WIN) break;
                    }
                }
            } else if (lane == 0) {            // status 2: the true path from the end of chain element c, serially
                State s = unpack(ws.flag[j0 + c] == 2 ? ws.ech[j0 + c] : ws.e1[j0 + c]);
                const BitSrc src = seg_src(ws, d, sg);
                status = 1;
                for (int j = c + 1; j < nk - 1; ++j) {
                    if (!advance(d, src, s, (uint32_t)(j + 1) * SUB_BITS, &cum)) { status = 3; break; }
                    c = j;
                    ws.ech[j0 + j] = pack(s);
                    ws.bch[j0 + j] = cum;
                    ws.flag[j0 + j] = 2;
                    if (pack(s) == ws.e1[j0 + j]) { status = 0; break; }   // path j is the true path from here on
                }
            }
            status = __shfl_sync(0xffffffffu, status, 0);
            c = __shfl_sync(0xffffffffu, c, 0);
            cum = __shfl_sync(0xffffffffu, cum, 0);
            __syncwarp();
        }
        if (status == 3 && lane == 0) fail(w, PN_JPEG_ERR_CODE);
    }
}

// ---- write: coefficients of the blocks that begin in each subsequence -------------------------------------------------------------
__global__ void __launch_bounds__(THREADS) write_kernel(Args a, Ws ws) {
    const long long total = ws.totals->nsub;
    for (long long j = blockIdx.x * (long long)THREADS + threadIdx.x; j < total; j += (long long)gridDim.x * THREADS) {
        const SubInfo info = ws.sub[j];
        if (info.img < 0) continue;
        ImgWs &w = ws.img[info.img];
        if (w.status != PN_JPEG_OK) continue;
        const pn_jpeg_desc &d = a.descs[info.img];
        const SegWs sg = ws.seg[info.seg];
        const BitSrc src = seg_src(ws, d, sg);
        const int s_idx = info.seg - w.seg_base;
        const long long nblocks = seg_blocks(d, s_idx);
        const bool last = info.k == info.nk - 1;
        const uint32_t end = (uint32_t)(info.k + 1) * SUB_BITS;
        // entry state: recomputed from the nearest chain element at or before subsequence k - 1 (the walk's flags)
        State s{0, 0, 0};
        uint32_t first = 0;
        if (info.k > 0) {
            const long long j0 = j - info.k;
            int c = info.k - 1;
            while (c > 0 && ws.flag[j0 + c] == 0) --c;
            const int f = ws.flag[j0 + c];
            const uint64_t e = f == 2 ? ws.ech[j0 + c] : ws.e1[j0 + c];
            if (f == 0 || e == kBadState) continue;
            s = unpack(e);
            first = ws.bch[j0 + c];
            if (c < info.k - 1 && !advance(d, src, s, (uint32_t)info.k * SUB_BITS, &first)) {
                fail(w, PN_JPEG_ERR_CODE);
                continue;
            }
        }
        if (s.z != 0 && !skip_rest_of_block(d, src, s)) {
            fail(w, PN_JPEG_ERR_CODE);
            continue;
        }
        long long blk = first;
        int16_t *coef = ws.coef + (w.blk_base + (long long)s_idx * d.restart_interval * d.blocks_per_mcu) * 64;
        bool ok = true;
        while (last ? blk < nblocks : s.pos < end) {
            if (blk >= nblocks) {
                fail(w, PN_JPEG_ERR_LENGTH);
                ok = false;
                break;
            }
            if (!decode_block(d, src, s, coef + blk * 64)) {
                fail(w, PN_JPEG_ERR_CODE);
                ok = false;
                break;
            }
            ++blk;
        }
        if (ok && last) {                      // the scan ends with the last block plus at most 7 padding bits
            const uint32_t bits = (sg.end - sg.start) * 8u;
            if (s.pos > bits || bits - s.pos > 7) fail(w, PN_JPEG_ERR_LENGTH);
        }
    }
}

// ---- progressive: one warp per image, the (scan, restart segment) pairs of each wave across the lanes ------------------------------
// The warp walks the scans of a wave in table order and cuts them at their RST markers (searched 32 bytes at a time), 32 segments
// per round; each lane then decodes its segment serially.  Waves are separated by __syncwarp, since a wave's scans refine the
// coefficients of the earlier ones.
__device__ int64_t warp_next_restart(const uint8_t *f, int64_t p, int64_t end, int lane) {
    for (int64_t b = p; b + 1 < end; b += 32) {
        const int64_t q = b + lane;
        const unsigned hit = __ballot_sync(0xffffffffu, q + 1 < end && f[q] == 0xFF && (f[q + 1] & 0xF8) == 0xD0);
        if (hit) return b + __ffs(hit) - 1;
    }
    return end;
}

__global__ void __launch_bounds__(32) progressive_kernel(Args a, Ws ws) {
    const int i = blockIdx.x, lane = threadIdx.x;
    const pn_jpeg_desc &d = a.descs[i];
    ImgWs &w = ws.img[i];
    if (d.kind != PN_JPEG_SUPPORTED_PROGRESSIVE || w.status != PN_JPEG_OK) return;
    const uint8_t *file = a.files + d.file_offset, *tab = a.files + scan_table_offset(d);
    const pn_jpeg_scans h = *reinterpret_cast<const pn_jpeg_scans *>(tab);
    const pn_jpeg_scan *sc = table_scans(tab);
    const pn_jpeg_huff *huff = table_huff(tab);
    int16_t *coef = ws.coef + w.blk_base * 64;
    for (long long j = lane; j < w.nblk * 8; j += 32) reinterpret_cast<uint4 *>(coef)[j] = make_uint4(0, 0, 0, 0);
    __syncwarp();
    int status = PN_JPEG_OK;
    for (int wave = 0; wave < h.n_waves && status == PN_JPEG_OK; ++wave) {
        int s = 0;
        while (s < h.n_scans && sc[s].wave != wave) ++s;
        int64_t p = s < h.n_scans ? sc[s].start : 0, k = 0;
        while (s < h.n_scans && status == PN_JPEG_OK) {
            int mine = -1;                     // this lane's pair: scan, segment, bytes
            int64_t my_k = 0, my_p = 0, my_e = 0;
            for (int n = 0; n < 32 && s < h.n_scans; ++n) {
                const pn_jpeg_scan &S = sc[s];
                const bool more = k + 1 < scan_segments(d, S);
                int64_t e = S.end;
                if (more) {
                    e = warp_next_restart(file, p, S.end, lane);
                    if (e == S.end || file[e + 1] != 0xD0 + (k & 7)) {
                        status = PN_JPEG_ERR_RESTART;
                        break;
                    }
                }
                if (lane == n) {
                    mine = s;
                    my_k = k;
                    my_p = p;
                    my_e = e;
                }
                if (more) {
                    p = e + 2;
                    ++k;
                } else {
                    do ++s; while (s < h.n_scans && sc[s].wave != wave);
                    p = s < h.n_scans ? sc[s].start : 0;
                    k = 0;
                }
            }
            int st = PN_JPEG_OK;
            if (status == PN_JPEG_OK && mine >= 0) {
                const pn_jpeg_scan &S = sc[mine];
                const int64_t units = scan_units(d, S), ri = S.restart_interval > 0 ? S.restart_interval : units;
                const int64_t u0 = my_k * ri;
                st = decode_scan_segment(d, S, huff, file, my_p, my_e, u0, units - u0 < ri ? units - u0 : ri, coef);
            }
            st = __reduce_min_sync(0xffffffffu, st);
            if (status == PN_JPEG_OK) status = st;
            __syncwarp();
        }
    }
    if (lane == 0 && status != PN_JPEG_OK) w.status = status;
}

// ---- DC: per-component running sums, one warp per segment ----------------------------------------------------------------------
__global__ void __launch_bounds__(THREADS) dc_kernel(Args a, Ws ws) {
    const int lane = threadIdx.x & 31;
    const long long warps = (long long)gridDim.x * (THREADS / 32);
    const long long total = ws.totals->nseg;
    for (long long sgi = blockIdx.x * (long long)(THREADS / 32) + (threadIdx.x >> 5); sgi < total; sgi += warps) {
        int lo = 0, hi = a.n_img - 1;
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (ws.img[mid].seg_base <= sgi) lo = mid; else hi = mid - 1;
        }
        const ImgWs &w = ws.img[lo];
        if (w.status != PN_JPEG_OK) continue;
        const pn_jpeg_desc &d = a.descs[lo];
        const int s_idx = (int)(sgi - w.seg_base);
        const long long n = seg_blocks(d, s_idx);
        int16_t *coef = ws.coef + (w.blk_base + (long long)s_idx * d.restart_interval * d.blocks_per_mcu) * 64;
        uint32_t carry[3] = {0, 0, 0};
        for (long long b0 = 0; b0 < n; b0 += 32) {
            const long long g = b0 + lane;
            const bool valid = g < n;
            const int comp = valid ? d.mcu_comp[g % d.blocks_per_mcu] : -1;
            const uint32_t v = valid ? (uint32_t)(int)coef[g * 64] : 0u;
            uint32_t outv = 0;
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                if (c >= d.ncomp) break;
                uint32_t x = comp == c ? v : 0u;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
                    if (lane >= o) x += y;
                }
                if (comp == c) outv = carry[c] + x;     // last_dc_val: int arithmetic done as unsigned, stored as JCOEF
                carry[c] += __shfl_sync(0xffffffffu, x, 31);
            }
            if (valid) coef[g * 64] = (int16_t)(uint16_t)outv;
        }
    }
}

// ---- IDCT: eight threads per block (pass 1: a column each; pass 2: a row each, the first ssize threads) --------------------------
__global__ void __launch_bounds__(THREADS) idct_kernel(Args a, Ws ws) {
    __shared__ int wsm[THREADS / 8][64];
    const int grp = threadIdx.x >> 3, r = threadIdx.x & 7;
    const long long total = ws.totals->nblk;
    for (long long g0 = blockIdx.x * (long long)(THREADS / 8); g0 < total; g0 += (long long)gridDim.x * (THREADS / 8)) {
        const long long gb = g0 + grp;
        int img = -1;
        if (gb < total) {
            int lo = 0, hi = a.n_img - 1;
            while (lo < hi) {
                const int mid = (lo + hi + 1) >> 1;
                if (ws.img[mid].blk_base <= gb) lo = mid; else hi = mid - 1;
            }
            img = ws.img[lo].status == PN_JPEG_OK ? lo : -1;
        }
        const pn_jpeg_desc *d = img >= 0 ? a.descs + img : nullptr;
        int comp = 0, bx = 0, by = 0, ss = 8;
        if (d) {
            block_place(*d, gb - ws.img[img].blk_base, &comp, &bx, &by);
            ss = comp_ssize(*d, a.denom, comp);
            idct_column_scaled(ws.coef + gb * 64, d->quant[comp], ss, r, wsm[grp]);
        }
        __syncwarp();
        if (d && ss == 8) {
            const int pitch = d->comp[comp].bw * 8;
            uint8_t o[8];
            idct_row(wsm[grp], r, o);
            uint8_t *dst = ws.planes + ws.img[img].plane_base[comp] + ((long long)by * 8 + r) * pitch + bx * 8;
            *reinterpret_cast<uint2 *>(dst) = make_uint2(o[0] | (o[1] << 8) | (o[2] << 16) | ((uint32_t)o[3] << 24),
                                                         o[4] | (o[5] << 8) | (o[6] << 16) | ((uint32_t)o[7] << 24));
        } else if (d && r < ss) {
            const int pitch = d->comp[comp].bw * ss;
            uint8_t o[4];
            idct_row_scaled(ws.coef + gb * 64, d->quant[comp], wsm[grp], ss, r, o);
            uint8_t *dst = ws.planes + ws.img[img].plane_base[comp] + ((long long)by * ss + r) * pitch + (long long)bx * ss;
            for (int c = 0; c < ss; ++c) dst[c] = o[c];
        }
        __syncwarp();
    }
}

// ---- colour: upsampling + YCbCr -> BGR into the frame rows, in the descriptor's orientation ---------------------------------------
constexpr int OT = 32;   // transposed orientations: OT x OT output tiles

__global__ void __launch_bounds__(THREADS) color_kernel(Args a, Ws ws) {
    __shared__ uint32_t tile[OT][OT + 1];
    const int i = blockIdx.y;
    const ImgWs &w = ws.img[i];
    const int st = w.status;
    const pn_jpeg_desc &d = a.descs[i];
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        a.status[i] = st;
        if (a.frame_hw) {                   // the frame at 1 / denom, oriented
            int oh = 0, ow = 0;
            if (st == PN_JPEG_OK)
                oriented_size(d.orientation, (d.height + a.denom - 1) / a.denom, (d.width + a.denom - 1) / a.denom, &oh, &ow);
            a.frame_hw[2 * i] = oh;
            a.frame_hw[2 * i + 1] = ow;
        }
    }
    if (st == PN_JPEG_SKIPPED || st == PN_JPEG_ERR_DESC) return;     // untouched: the host's frame, or no trusted size
    Scaled g;
    scaled_geometry(d, a.denom, &g);       // plan_kernel checked it and the orientation
    const int H = g.h, W = g.w, o = d.orientation;                 // H x W: the decoded frame
    int OH, OW;
    oriented_size(o, H, W, &OH, &OW);
    uint8_t *frame = a.frames + (long long)i * a.stride;
    const uint8_t *plane[3];
    int pitch[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {           // components past ncomp are never read
        plane[c] = ws.planes + w.plane_base[c];
        pitch[c] = d.comp[c].bw * g.comp[c].ssize;
    }
    if (st == PN_JPEG_OK && orient_transposes(o)) {
        // An output row is a source column.  Phase 1 walks the tile's source rows (a warp on 32 consecutive source pixels, i.e. one
        // output column) into tile[output row][output column]; phase 2 writes the output rows.  Row stride OT + 1: no bank conflicts.
        const int tiles_x = (OW + OT - 1) / OT, ntiles = tiles_x * ((OH + OT - 1) / OT);
        for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
            const int ty0 = (t / tiles_x) * OT, tx0 = (t % tiles_x) * OT;
            for (int k = threadIdx.x; k < OT * OT; k += THREADS) {
                const int ty = k % OT, tx = k / OT, y = ty0 + ty, x = tx0 + tx;
                if (y < OH && x < OW) {
                    int sy, sx;
                    uint8_t bgr[3];
                    orient_source(o, H, W, y, x, &sy, &sx);
                    pixel_bgr(d, g, plane, pitch, sy, sx, bgr);
                    tile[ty][tx] = bgr[0] | (bgr[1] << 8) | ((uint32_t)bgr[2] << 16);
                }
            }
            __syncthreads();
            for (int k = threadIdx.x; k < OT * OT; k += THREADS) {
                const int ty = k / OT, tx = k % OT, y = ty0 + ty, x = tx0 + tx;
                if (y < OH && x < OW) {
                    const uint32_t v = tile[ty][tx];
                    uint8_t *px = frame + 3 * ((long long)y * OW + x);
                    px[0] = (uint8_t)v;
                    px[1] = (uint8_t)(v >> 8);
                    px[2] = (uint8_t)(v >> 16);
                }
            }
            __syncthreads();
        }
        return;
    }
    const long long npx = (long long)OH * OW;
    for (long long p = blockIdx.x * (long long)THREADS + threadIdx.x; p < npx; p += (long long)gridDim.x * THREADS) {
        uint8_t bgr[3] = {0, 0, 0};
        if (st == PN_JPEG_OK) {
            int y = (int)(p / OW), x = (int)(p % OW);
            if (o > 1) orient_source(o, H, W, y, x, &y, &x);   // flips keep the row order
            pixel_bgr(d, g, plane, pitch, y, x, bgr);
        }
        frame[3 * p] = bgr[0];
        frame[3 * p + 1] = bgr[1];
        frame[3 * p + 2] = bgr[2];
    }
}

Ws bind(void *base, const Layout &L) {
    char *b = static_cast<char *>(base);
    Ws w;
    w.totals = reinterpret_cast<Totals *>(b + L.totals);
    w.img = reinterpret_cast<ImgWs *>(b + L.img);
    w.seg = reinterpret_cast<SegWs *>(b + L.seg);
    w.sub = reinterpret_cast<SubInfo *>(b + L.sub);
    w.e1 = reinterpret_cast<uint64_t *>(b + L.e1);
    w.ech = reinterpret_cast<uint64_t *>(b + L.ech);
    w.m = reinterpret_cast<int *>(b + L.m);
    w.flag = reinterpret_cast<int *>(b + L.flag);
    w.c1 = reinterpret_cast<uint32_t *>(b + L.c1);
    w.c2 = reinterpret_cast<uint32_t *>(b + L.c2);
    w.bch = reinterpret_cast<uint32_t *>(b + L.bch);
    w.coef = reinterpret_cast<int16_t *>(b + L.coef);
    w.planes = reinterpret_cast<uint8_t *>(b + L.planes);
    w.ds = reinterpret_cast<uint8_t *>(b + L.ds);
    w.nseg_cap = L.nseg_cap;
    w.nsub_cap = L.nsub_cap;
    w.nblk_cap = L.nblk_cap;
    return w;
}

// max_h x max_w: the full-size capacity (scale_denom times the output capacity)
bool caps_ok(int n_img, int64_t arena_bytes, long long max_h, long long max_w) {
    return n_img > 0 && n_img <= 65535 && arena_bytes > 0 && arena_bytes < (1ll << 40) && max_h > 0 && max_w > 0 &&
           max_h <= 65500 && max_w <= 65500;
}

}  // namespace
}  // namespace pn

using namespace pn;

extern "C" int pn_jpeg_workspace_scaled(int n_img, int64_t arena_bytes, int max_h, int max_w, int scale_denom,
                                        size_t *bytes_host) {
    PN_CHECK_ARG(bytes_host, "pn_jpeg_workspace_scaled: null pointer");
    PN_CHECK_ARG(valid_denom(scale_denom), "pn_jpeg_workspace_scaled: scale_denom %d is not 1, 2, 4 or 8", scale_denom);
    PN_CHECK_ARG(caps_ok(n_img, arena_bytes, (long long)max_h * scale_denom, (long long)max_w * scale_denom),
                 "pn_jpeg_workspace_scaled: bad capacity (%d images, %lld bytes, %d x %d at 1/%d)", n_img, (long long)arena_bytes,
                 max_h, max_w, scale_denom);
    *bytes_host = layout(n_img, arena_bytes, max_h * scale_denom, max_w * scale_denom).bytes;
    return PN_OK;
}

extern "C" int pn_jpeg_workspace(int n_img, int64_t arena_bytes, int max_h, int max_w, size_t *bytes_host) {
    return pn_jpeg_workspace_scaled(n_img, arena_bytes, max_h, max_w, 1, bytes_host);
}

extern "C" int pn_jpeg_decode_scaled(const uint8_t *files, int64_t arena_bytes, const pn_jpeg_desc *descs, int n_img, int max_h,
                                     int max_w, int scale_denom, uint8_t *frames, int64_t frame_stride, int *frame_hw,
                                     void *workspace, size_t ws_bytes, int *status, pn_stream_t stream) {
    PN_CHECK_ARG(files && descs && frames && workspace && status, "pn_jpeg_decode_scaled: null pointer");
    PN_CHECK_ARG(valid_denom(scale_denom), "pn_jpeg_decode_scaled: scale_denom %d is not 1, 2, 4 or 8", scale_denom);
    PN_CHECK_ARG(caps_ok(n_img, arena_bytes, (long long)max_h * scale_denom, (long long)max_w * scale_denom),
                 "pn_jpeg_decode_scaled: bad capacity (%d images, %lld bytes, %d x %d at 1/%d)", n_img, (long long)arena_bytes,
                 max_h, max_w, scale_denom);
    PN_CHECK_ARG(frame_stride >= 3ll * max_h * max_w, "pn_jpeg_decode_scaled: frame_stride %lld < 3 * max_h * max_w",
                 (long long)frame_stride);
    PN_CHECK_ARG(((uintptr_t)workspace & 255) == 0, "pn_jpeg_decode_scaled: workspace must be 256-byte aligned");
    const Layout L = layout(n_img, arena_bytes, max_h * scale_denom, max_w * scale_denom);
    PN_CHECK_ARG(ws_bytes >= L.bytes, "pn_jpeg_decode_scaled: workspace %zu < %zu bytes (pn_jpeg_workspace_scaled)", ws_bytes,
                 L.bytes);
    Args a{files, arena_bytes, descs, n_img, max_h, max_w, scale_denom, frames, frame_stride, frame_hw, status};
    const Ws w = bind(workspace, L);
    const cudaStream_t st = as_stream(stream);
    const int grid = 4 * num_sms();
    plan_kernel<<<n_img, 32, 0, st>>>(a, w);
    PN_CHECK_LAUNCH();
    layout_kernel<<<1, THREADS, 0, st>>>(a, w);
    PN_CHECK_LAUNCH();
    destuff_kernel<<<n_img, THREADS, 0, st>>>(a, w);
    PN_CHECK_LAUNCH();
    spec_kernel<<<grid, THREADS, 0, st>>>(a, w);
    PN_CHECK_LAUNCH();
    merge_kernel<<<grid, THREADS, 0, st>>>(a, w);
    PN_CHECK_LAUNCH();
    walk_kernel<<<grid, THREADS, 0, st>>>(a, w);
    PN_CHECK_LAUNCH();
    write_kernel<<<grid, THREADS, 0, st>>>(a, w);
    PN_CHECK_LAUNCH();
    progressive_kernel<<<n_img, 32, 0, st>>>(a, w);
    PN_CHECK_LAUNCH();
    dc_kernel<<<grid, THREADS, 0, st>>>(a, w);
    PN_CHECK_LAUNCH();
    idct_kernel<<<grid, THREADS, 0, st>>>(a, w);
    PN_CHECK_LAUNCH();
    const long long px = (long long)max_h * max_w;
    long long gx = (px + THREADS * 4 - 1) / (THREADS * 4);
    if (gx > 1024) gx = 1024;
    color_kernel<<<dim3((unsigned)gx, (unsigned)n_img), THREADS, 0, st>>>(a, w);
    PN_CHECK_LAUNCH();
    return PN_OK;
}

extern "C" int pn_jpeg_decode(const uint8_t *files, int64_t arena_bytes, const pn_jpeg_desc *descs, int n_img, int max_h, int max_w,
                              uint8_t *frames, int64_t frame_stride, int *frame_hw, void *workspace, size_t ws_bytes, int *status,
                              pn_stream_t stream) {
    return pn_jpeg_decode_scaled(files, arena_bytes, descs, n_img, max_h, max_w, 1, frames, frame_stride, frame_hw, workspace,
                                 ws_bytes, status, stream);
}
