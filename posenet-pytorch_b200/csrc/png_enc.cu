// pn_png_encode: uint8 BGR frames on the device -> PNG files, bit-exact with cv2.imencode(".png") (arithmetic: png_encode.cuh).
//
// One call encodes a batch in ten launches (and one memset) whose geometry depends only on the capacity (n_img, max_h, max_w),
// so the call can be captured in a CUDA graph.  The filtered image of frame i is its n_i = h_i (3 w_i + 1) bytes, cut into
// tiles of TILE bytes:
//   filter   a CTA per tile: the SUB-filtered bytes, the tile's first and last run start, Adler-32 partial sums
//   carry    a CTA per image: for every tile, the last run start before it and the first run start after it
//   count    a CTA per tile: every byte learns its run (start, end) from its neighbours and the carries; the tile's symbols
//   scan     a CTA per image: exclusive sum of the tiles' symbol counts
//   symbols  a CTA per tile: as count, then writes each symbol (literal or match length) at its index, and the bytes where
//            blocks of 16383 symbols start and where their last symbol starts
//   trees    a CTA per block: the block's histogram; one thread runs trees.c (build_tree x 3, the block-type choice)
//   place    one CTA: a thread per image lays its blocks out (stored blocks byte-align, so a block's size depends on where it
//            starts), the file sizes, their exclusive sum into out_offsets
//   clear    a grid-stride loop zeroes the words each image's deflate stream uses
//   emit     a CTA per block: the header by one thread, the symbols by all (bit positions from a CTA scan), stored blocks as
//            bytes; words shared with a neighbour by atomicOr into a stream cleared beforehand
//   pack     a CTA per IDAT chunk: length, type, payload (zlib header, deflate bytes, Adler-32), CRC-32 of 256 pieces combined
//            by crc32_combine; the first chunk's CTA writes the signature and IHDR, the last one's IEND
#include <limits.h>

#include "common.cuh"
#include "png_encode.cuh"

namespace pn {
namespace {

using namespace pnge;

constexpr int THREADS = 256;
constexpr int BPT = 16;                           // bytes per thread in the tile kernels
constexpr int TILE = THREADS * BPT;
constexpr int CTA_THREADS = 1024;                 // the per-image kernels
constexpr int PACK_BPT = (4 + kIdat + THREADS - 1) / THREADS;   // CRC input bytes ("IDAT" + payload) per thread in pack
constexpr int NONE = -1;

struct Args {
    const uint8_t *frames;
    int n_img, max_h, max_w;
    int64_t stride;
    const int *frame_hw;
    uint8_t *out;
    int64_t *offsets;
};

struct Block {
    BlockCode c;
    unsigned long long pos;                       // first bit in the image's deflate stream
    uint32_t b0, b1;                              // bytes [b0, b1) of the filtered image
};

struct Layout {
    size_t filt, sym, tfirst, tlast, tcarry_a, tcarry_e, tcount, bstart, blast, blocks, nsym, adler, dbytes, size, words, bytes;
    long long ncap, tcap, bcap, wcap, ccap;
};

size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

Layout layout(int n_img, int max_h, int max_w) {
    Layout L;
    L.ncap = data_size(max_h, max_w);
    L.tcap = (L.ncap + TILE - 1) / TILE;
    L.bcap = max_blocks(L.ncap);
    L.wcap = (deflate_bound(L.ncap) + 3) / 4 + 1;
    L.ccap = num_chunks(zlib_bound(L.ncap));
    size_t o = 0;
    auto take = [&](size_t bytes) { const size_t at = o; o = align256(o + bytes); return at; };
    L.filt = take((size_t)n_img * L.ncap);
    L.sym = take(2ull * n_img * L.ncap);
    L.tfirst = take(4ull * n_img * L.tcap);
    L.tlast = take(4ull * n_img * L.tcap);
    L.tcarry_a = take(4ull * n_img * L.tcap);
    L.tcarry_e = take(4ull * n_img * L.tcap);
    L.tcount = take(4ull * n_img * L.tcap);
    L.bstart = take(4ull * n_img * L.bcap);
    L.blast = take(4ull * n_img * L.bcap);
    L.blocks = take(sizeof(Block) * n_img * L.bcap);
    L.nsym = take(4ull * n_img);
    L.adler = take(16ull * n_img);
    L.dbytes = take(8ull * n_img);
    L.size = take(8ull * n_img);
    L.words = take(4ull * n_img * L.wcap);
    L.bytes = o;
    return L;
}

struct Ws {
    uint8_t *filt;
    uint16_t *sym;        // per symbol: a literal (0..255) or 256 + match length - 3
    int *tfirst, *tlast;  // per tile: first / last run start in it (NONE)
    int *tcarry_a;        // per tile: the last run start before it
    int *tcarry_e;        // per tile: the first run start after it (n when none)
    uint32_t *tcount;     // per tile: symbols (count), then the index of its first symbol (scan)
    uint32_t *bstart;     // per block: the byte its first symbol starts at
    uint32_t *blast;      // per block: the byte its last symbol starts at
    Block *blocks;
    uint32_t *nsym;
    unsigned long long *adler;   // per image: sum of the bytes, sum of (n - p) * byte, both mod 65521
    long long *dbytes;    // per image: deflate stream bytes
    long long *size;      // file sizes
    uint32_t *words;      // deflate streams, LSB-first bit order in little-endian words
    long long ncap, tcap, bcap, wcap, ccap;
};

Ws bind(void *base, const Layout &L) {
    char *b = static_cast<char *>(base);
    Ws w;
    w.filt = reinterpret_cast<uint8_t *>(b + L.filt);
    w.sym = reinterpret_cast<uint16_t *>(b + L.sym);
    w.tfirst = reinterpret_cast<int *>(b + L.tfirst);
    w.tlast = reinterpret_cast<int *>(b + L.tlast);
    w.tcarry_a = reinterpret_cast<int *>(b + L.tcarry_a);
    w.tcarry_e = reinterpret_cast<int *>(b + L.tcarry_e);
    w.tcount = reinterpret_cast<uint32_t *>(b + L.tcount);
    w.bstart = reinterpret_cast<uint32_t *>(b + L.bstart);
    w.blast = reinterpret_cast<uint32_t *>(b + L.blast);
    w.blocks = reinterpret_cast<Block *>(b + L.blocks);
    w.nsym = reinterpret_cast<uint32_t *>(b + L.nsym);
    w.adler = reinterpret_cast<unsigned long long *>(b + L.adler);
    w.dbytes = reinterpret_cast<long long *>(b + L.dbytes);
    w.size = reinterpret_cast<long long *>(b + L.size);
    w.words = reinterpret_cast<uint32_t *>(b + L.words);
    w.ncap = L.ncap, w.tcap = L.tcap, w.bcap = L.bcap, w.wcap = L.wcap, w.ccap = L.ccap;
    return w;
}

// Image i's size: its own with frame_hw (a size outside 1..max is an empty file), else max_h x max_w.
__device__ __forceinline__ void image_hw(const Args &a, int i, int *h, int *w) {
    *h = a.max_h, *w = a.max_w;
    if (a.frame_hw) {
        *h = a.frame_hw[2 * i];
        *w = a.frame_hw[2 * i + 1];
        if (*h < 1 || *w < 1 || *h > a.max_h || *w > a.max_w) *h = *w = 0;
    }
}

__device__ __forceinline__ long long image_n(const Args &a, int i) {
    int h, w;
    image_hw(a, i, &h, &w);
    return data_size(h, w);
}

// ---- CTA scans ---------------------------------------------------------------------------------------------------------------
// Exclusive scan of v over the CTA (blockDim.x threads, a multiple of 32) under op with identity id; *total: the reduction.
template <typename T, typename Op>
__device__ T cta_exclusive(T v, T id, Op op, T *total, T *sm) {   // sm: 33 entries
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    T x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const T y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x = op(y, x);
    }
    if (lane == 31) sm[warp] = x;
    __syncthreads();
    if (warp == 0) {
        const T t = lane < nw ? sm[lane] : id;
        T s = t;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const T y = __shfl_up_sync(0xffffffffu, s, o);
            if (lane >= o) s = op(y, s);
        }
        if (lane < nw) sm[lane] = s;                              // inclusive over warps
        if (lane == 31) sm[32] = s;
    }
    __syncthreads();
    const T before_warp = warp ? sm[warp - 1] : id;
    T excl = __shfl_up_sync(0xffffffffu, x, 1);
    if (lane == 0) excl = id;
    const T r = op(before_warp, excl);
    *total = sm[32];
    __syncthreads();
    return r;
}

struct Add { template <typename T> __device__ T operator()(T a, T b) const { return a + b; } };
struct Max { __device__ int operator()(int a, int b) const { return a > b ? a : b; } };
struct Min { __device__ int operator()(int a, int b) const { return a < b ? a : b; } };

// ---- filter: a CTA per tile ------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(THREADS) filter_kernel(Args a, Ws ws) {
    __shared__ int sm[33];
    const int i = (int)(blockIdx.x / ws.tcap), t = (int)(blockIdx.x - (long long)i * ws.tcap);
    int h, w;
    image_hw(a, i, &h, &w);
    const long long n = data_size(h, w);
    if ((long long)t * TILE >= n) return;
    const uint8_t *frame = a.frames + (long long)i * a.stride;
    uint8_t *filt = ws.filt + (long long)i * ws.ncap;
    const long long p0 = (long long)t * TILE + threadIdx.x * BPT;
    int first = INT_MAX, last = NONE;
    unsigned long long s1 = 0, s2 = 0;
    if (p0 < n) {
        uint8_t prev = p0 ? filtered_byte(frame, w, p0 - 1) : 0;
        for (int k = 0; k < BPT && p0 + k < n; k++) {
            const long long p = p0 + k;
            const uint8_t v = filtered_byte(frame, w, p);
            filt[p] = v;
            if (p == 0 || v != prev) {
                if (first == INT_MAX) first = (int)p;
                last = (int)p;
            }
            prev = v;
            s1 += v;
            s2 += (unsigned long long)(n - p) * v;
        }
    }
    s1 = __reduce_add_sync(0xffffffffu, (unsigned)s1);
#pragma unroll
    for (int o = 16; o; o >>= 1) s2 += __shfl_xor_sync(0xffffffffu, s2, o);
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(ws.adler + 2 * i, s1 % kAdlerBase);
        atomicAdd(ws.adler + 2 * i + 1, s2 % kAdlerBase);
    }
    int tot;
    cta_exclusive<int>(first, INT_MAX, Min(), &tot, sm);
    if (threadIdx.x == 0) ws.tfirst[(long long)i * ws.tcap + t] = tot;
    cta_exclusive<int>(last, NONE, Max(), &tot, sm);
    if (threadIdx.x == 0) ws.tlast[(long long)i * ws.tcap + t] = tot;
}

// ---- carry: a CTA per image -------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(CTA_THREADS) carry_kernel(Args a, Ws ws) {
    __shared__ int sm[33];
    const int i = blockIdx.x;
    const long long n = image_n(a, i);
    const int nt = (int)((n + TILE - 1) / TILE);
    const int *tf = ws.tfirst + (long long)i * ws.tcap, *tl = ws.tlast + (long long)i * ws.tcap;
    int *ca = ws.tcarry_a + (long long)i * ws.tcap, *ce = ws.tcarry_e + (long long)i * ws.tcap;
    int run = NONE;
    for (int t0 = 0; t0 < nt; t0 += CTA_THREADS) {                 // last start before each tile
        const int t = t0 + threadIdx.x;
        int tot;
        const int e = cta_exclusive<int>(t < nt ? tl[t] : NONE, NONE, Max(), &tot, sm);
        if (t < nt) ca[t] = e > run ? e : run;
        run = tot > run ? tot : run;
    }
    run = (int)n;
    for (int t0 = 0; t0 < nt; t0 += CTA_THREADS) {                 // first start after each tile: the scan from the end
        const int t = nt - 1 - (t0 + threadIdx.x);
        int tot;
        const int e = cta_exclusive<int>(t >= 0 ? (tf[t] == INT_MAX ? (int)n : tf[t]) : (int)n, (int)n, Min(), &tot, sm);
        if (t >= 0) ce[t] = e < run ? e : run;
        run = tot < run ? tot : run;
    }
}

// ---- count / symbols: a CTA per tile ------------------------------------------------------------------------------------------
template <bool WRITE>
__global__ void __launch_bounds__(THREADS) symbols_kernel(Args a, Ws ws) {
    __shared__ int sm[33];
    __shared__ uint32_t su[33];
    __shared__ int snext[THREADS];
    const int i = (int)(blockIdx.x / ws.tcap), t = (int)(blockIdx.x - (long long)i * ws.tcap);
    const long long n = image_n(a, i);
    if ((long long)t * TILE >= n) return;
    const uint8_t *filt = ws.filt + (long long)i * ws.ncap;
    const long long p0 = (long long)t * TILE + threadIdx.x * BPT;
    const int cnt = p0 < n ? (int)(n - p0 < BPT ? n - p0 : BPT) : 0;
    uint8_t v[BPT];
    uint32_t starts = 0;                                             // bit k: byte p0 + k starts a run
    int first = INT_MAX, last = NONE;
    uint8_t prev = cnt && p0 ? filt[p0 - 1] : 0;
#pragma unroll
    for (int k = 0; k < BPT; k++) {
        v[k] = k < cnt ? filt[p0 + k] : 0;
        if (k < cnt && (p0 + k == 0 || v[k] != prev)) {
            starts |= 1u << k;
            if (first == INT_MAX) first = (int)(p0 + k);
            last = (int)(p0 + k);
        }
        prev = v[k];
    }
    const long long tc = (long long)i * ws.tcap + t;
    int tot;
    int ra = cta_exclusive<int>(last, NONE, Max(), &tot, sm);       // the last run start before this thread's bytes
    if (ra == NONE) ra = ws.tcarry_a[tc];
    // the first run start after this thread's bytes: an exclusive min-scan in reverse thread order
    snext[threadIdx.x] = first;
    __syncthreads();
    const int mirrored = snext[THREADS - 1 - threadIdx.x];
    __syncthreads();
    const int after = cta_exclusive<int>(mirrored, INT_MAX, Min(), &tot, sm);
    snext[THREADS - 1 - threadIdx.x] = after;
    __syncthreads();
    int e = snext[threadIdx.x] == INT_MAX ? ws.tcarry_e[tc] : snext[threadIdx.x];
    // each byte's run: from the last start at or before it to the first start after it
    int ends[BPT];
#pragma unroll
    for (int k = BPT - 1; k >= 0; k--) {
        ends[k] = e;
        if (starts >> k & 1) e = (int)(p0 + k);
    }
    uint32_t nsym = 0;
    int lcs[BPT];
    int s = ra;
#pragma unroll
    for (int k = 0; k < BPT; k++) {
        if (starts >> k & 1) s = (int)(p0 + k);
        int lc;
        lcs[k] = k < cnt && run_symbol_at(p0 + k - s, ends[k] - s, v[k], &lc) ? lc : NONE;
        nsym += lcs[k] != NONE;
    }
    uint32_t total;
    const uint32_t before = cta_exclusive<uint32_t>(nsym, 0u, Add(), &total, su);
    if (!WRITE) {
        if (threadIdx.x == 0) ws.tcount[tc] = total;
        return;
    }
    uint32_t idx = ws.tcount[tc] + before;
    uint16_t *sym = ws.sym + (long long)i * ws.ncap;
    uint32_t *bstart = ws.bstart + (long long)i * ws.bcap, *blast = ws.blast + (long long)i * ws.bcap;
#pragma unroll
    for (int k = 0; k < BPT; k++) {
        if (lcs[k] == NONE) continue;
        sym[idx] = (uint16_t)lcs[k];
        const uint32_t r = idx % kBlockSyms;
        if (r == 0) bstart[idx / kBlockSyms] = (uint32_t)(p0 + k);
        if (r == kBlockSyms - 1) blast[idx / kBlockSyms] = (uint32_t)(p0 + k);
        idx++;
    }
}

// ---- scan: a CTA per image --------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(CTA_THREADS) scan_kernel(Args a, Ws ws) {
    __shared__ uint32_t sm[33];
    const int i = blockIdx.x;
    const long long n = image_n(a, i);
    const int nt = (int)((n + TILE - 1) / TILE);
    uint32_t *tc = ws.tcount + (long long)i * ws.tcap;
    uint32_t run = 0;
    for (int t0 = 0; t0 < nt; t0 += CTA_THREADS) {
        const int t = t0 + threadIdx.x;
        uint32_t tot;
        const uint32_t e = cta_exclusive<uint32_t>(t < nt ? tc[t] : 0u, 0u, Add(), &tot, sm);
        if (t < nt) tc[t] = e + run;
        run += tot;
    }
    if (threadIdx.x == 0) ws.nsym[i] = run;
}

__device__ __forceinline__ long long num_blocks(long long n, uint32_t nsym) { return n ? nsym / kBlockSyms + 1 : 0; }

// ---- trees: a CTA per block ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(THREADS) trees_kernel(Args a, Ws ws) {
    __shared__ uint32_t hist[L_CODES + 1];        // [L_CODES]: matches
    __shared__ FlushWork work;
    const int i = (int)(blockIdx.x / ws.bcap);
    const long long b = blockIdx.x - (long long)i * ws.bcap;
    const long long n = image_n(a, i);
    const uint32_t S = ws.nsym[i];
    const long long nb = num_blocks(n, S);
    if (b >= nb) return;
    for (int k = threadIdx.x; k <= L_CODES; k += THREADS) hist[k] = 0;
    __syncthreads();
    const long long s0 = b * kBlockSyms, s1 = s0 + kBlockSyms < S ? s0 + kBlockSyms : S;
    const uint16_t *sym = ws.sym + (long long)i * ws.ncap;
    for (long long s = s0 + threadIdx.x; s < s1; s += THREADS) {
        const int lc = sym[s];
        if (lc < 256) atomicAdd(&hist[lc], 1u);
        else {
            atomicAdd(&hist[length_code(lc - 256) + LITERALS + 1], 1u);
            atomicAdd(&hist[L_CODES], 1u);
        }
    }
    __syncthreads();
    if (threadIdx.x) return;
    const uint32_t *bstart = ws.bstart + (long long)i * ws.bcap, *blast = ws.blast + (long long)i * ws.bcap;
    const bool last = b == nb - 1;
    const long long B = s0 < S ? bstart[b] : n, E = s1 < S ? bstart[b + 1] : n, P = last ? n : blast[b];
    const int wbits = window_bits(n);
    Block *blk = ws.blocks + (long long)i * ws.bcap + b;
    flush_block(hist, hist[L_CODES], E - B, B >= slides_before(P, n, wbits) << wbits, work, &blk->c);
    blk->b0 = (uint32_t)B;
    blk->b1 = (uint32_t)E;
}

// Block b's bits from its first (type) bit, given the bit it starts at.
__device__ __forceinline__ unsigned long long block_bits(const Block &blk, unsigned long long pos) {
    if (blk.c.type != STORED) return (unsigned long long)blk.c.bits;
    const unsigned long long aligned = (pos + 3 + 7) & ~7ull;
    return aligned - pos + 32 + 8ull * (blk.b1 - blk.b0);
}

// ---- place: one CTA ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(CTA_THREADS) place_kernel(Args a, Ws ws) {
    __shared__ long long sm[33];
    long long run = 0;
    for (int i0 = 0; i0 < a.n_img; i0 += CTA_THREADS) {
        const int i = i0 + threadIdx.x;
        long long size = 0;
        if (i < a.n_img) {
            const long long n = image_n(a, i), nb = num_blocks(n, ws.nsym[i]);
            unsigned long long pos = 0;
            Block *blk = ws.blocks + (long long)i * ws.bcap;
            for (long long b = 0; b < nb; b++) {
                blk[b].pos = pos;
                pos += block_bits(blk[b], pos);
            }
            const long long db = (long long)((pos + 7) / 8);
            ws.dbytes[i] = db;
            size = n ? file_size(2 + db + 4) : 0;
            ws.size[i] = size;
        }
        long long tot;
        const long long o = cta_exclusive<long long>(size, 0ll, Add(), &tot, sm) + run;
        if (i < a.n_img) a.offsets[i] = o;
        run += tot;
    }
    if (threadIdx.x == 0) a.offsets[a.n_img] = run;
}

// ---- clear: the words each stream uses ----------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(THREADS) clear_kernel(Args a, Ws ws) {
    const long long total = (long long)a.n_img * ws.wcap;
    for (long long k = blockIdx.x * (long long)THREADS + threadIdx.x; k < total; k += (long long)gridDim.x * THREADS) {
        const int i = (int)(k / ws.wcap);
        const long long wi = k - (long long)i * ws.wcap;
        if (wi < (ws.dbytes[i] + 3) / 4) ws.words[k] = 0;
    }
}

// ---- emit: a CTA per block -----------------------------------------------------------------------------------------------------------
struct WordSink {                                 // send_bits into a cleared word stream from bit pos on
    uint32_t *words;
    unsigned long long wi, acc;
    int fill;
    bool first;
    __device__ WordSink(uint32_t *w, unsigned long long pos) : words(w), wi(pos >> 5), acc(0), fill((int)(pos & 31)), first(true) {}
    __device__ __forceinline__ void operator()(uint32_t v, int n) {
        acc |= (unsigned long long)(v & ((1u << n) - 1u)) << fill;
        fill += n;
        if (fill >= 32) {
            if (first) atomicOr(words + wi, (uint32_t)acc);
            else words[wi] = (uint32_t)acc;
            first = false;
            ++wi;
            acc >>= 32;
            fill -= 32;
        }
    }
    __device__ __forceinline__ void finish() {
        if (fill) atomicOr(words + wi, (uint32_t)acc);           // shared with what follows
    }
};

__global__ void __launch_bounds__(THREADS) emit_kernel(Args a, Ws ws) {
    __shared__ BlockCode bc;
    __shared__ unsigned long long s_hdr;
    __shared__ unsigned long long sm[33];
    const int i = (int)(blockIdx.x / ws.bcap);
    const long long b = blockIdx.x - (long long)i * ws.bcap;
    const long long n = image_n(a, i);
    const uint32_t S = ws.nsym[i];
    const long long nb = num_blocks(n, S);
    if (b >= nb) return;
    const Block *blk = ws.blocks + (long long)i * ws.bcap + b;
    {
        const uint32_t *src = reinterpret_cast<const uint32_t *>(&blk->c);
        uint32_t *dst = reinterpret_cast<uint32_t *>(&bc);
        static_assert(sizeof(BlockCode) % 4 == 0, "BlockCode is copied as words");
        for (int k = threadIdx.x; k < (int)(sizeof(BlockCode) / 4); k += THREADS) dst[k] = src[k];
    }
    __syncthreads();
    uint32_t *words = ws.words + (long long)i * ws.wcap;
    const unsigned long long pos = blk->pos;
    const bool last = b == nb - 1;
    if (threadIdx.x == 0) {
        WordSink sink(words, pos);
        send_block_header(bc, last, sink);
        sink.finish();
        CountBits cb;
        send_block_header(bc, last, cb);
        s_hdr = (unsigned long long)cb.bits;
    }
    if (bc.type == STORED) {
        // LEN, NLEN and the bytes from the byte after the 3-bit header
        const unsigned long long at = (pos + 3 + 7) / 8;
        const uint32_t len = blk->b1 - blk->b0;
        const uint8_t *src = ws.filt + (long long)i * ws.ncap + blk->b0;
        const unsigned long long end = at + 4 + len;
        for (unsigned long long wk = at / 4 + threadIdx.x; wk * 4 < end; wk += THREADS) {
            uint32_t word = 0;
            bool whole = true;
            for (int j = 0; j < 4; j++) {
                const unsigned long long k = wk * 4 + j;
                if (k < at || k >= end) { whole = false; continue; }
                const unsigned long long o = k - at;
                const uint32_t byte = o < 2 ? (len >> (8 * o)) & 0xFF : o < 4 ? (~len >> (8 * (o - 2))) & 0xFF : src[o - 4];
                word |= byte << (8 * j);
            }
            if (whole) words[wk] = word;
            else atomicOr(words + wk, word);
        }
        return;
    }
    __syncthreads();
    const long long s0 = b * kBlockSyms, s1 = s0 + kBlockSyms < S ? s0 + kBlockSyms : S;
    const long long per = (s1 - s0 + THREADS - 1) / THREADS;
    const long long m0 = s0 + threadIdx.x * per, m1 = m0 + per < s1 ? m0 + per : s1;
    const uint16_t *sym = ws.sym + (long long)i * ws.ncap;
    unsigned long long bits = 0;
    for (long long s = m0; s < m1; s++) bits += symbol_bits(bc, sym[s]);
    unsigned long long tot;
    const unsigned long long before = cta_exclusive<unsigned long long>(bits, 0ull, Add(), &tot, sm);
    const unsigned long long body = pos + s_hdr;
    if (m0 < m1) {
        WordSink sink(words, body + before);
        for (long long s = m0; s < m1; s++) send_symbol(bc, sym[s], sink);
        sink.finish();
    }
    if (threadIdx.x == 0) {
        WordSink sink(words, body + tot);
        sink(bc.code[END_BLOCK], bc.len[END_BLOCK]);
        sink.finish();
    }
}

// ---- pack: a CTA per IDAT chunk ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint8_t zlib_byte(const uint8_t *zh, const uint32_t *words, long long db, uint32_t adler, long long k) {
    if (k < 2) return zh[k];
    k -= 2;
    if (k < db) return (uint8_t)(words[k >> 2] >> (8 * (k & 3)));
    return (uint8_t)(adler >> (24 - 8 * (k - db)));
}

__global__ void __launch_bounds__(THREADS) pack_kernel(Args a, Ws ws) {
    __shared__ uint32_t table[256];
    __shared__ uint32_t scrc[THREADS];
    __shared__ long long slen[THREADS];
    const int i = (int)(blockIdx.x / ws.ccap);
    const long long c = blockIdx.x - (long long)i * ws.ccap;
    int h, w;
    image_hw(a, i, &h, &w);
    const long long n = data_size(h, w);
    if (!n) return;
    const long long db = ws.dbytes[i], zlen = 2 + db + 4, nc = num_chunks(zlen);
    if (c >= nc) return;
    {
        uint32_t r = threadIdx.x;
        for (int k = 0; k < 8; k++) r = r & 1 ? (r >> 1) ^ kCrcPoly : r >> 1;
        table[threadIdx.x] = r;
    }
    uint8_t zh[2];
    zlib_header(n, window_bits(n), zh);
    const uint32_t adler = (uint32_t)(((ws.adler[2 * i + 1] + n) % kAdlerBase) << 16 | ((ws.adler[2 * i] + 1) % kAdlerBase));
    uint8_t *o = a.out + a.offsets[i];
    if (c == 0 && threadIdx.x == 0) write_head(h, w, o);
    if (c == nc - 1 && threadIdx.x == 0) write_tail(o + ws.size[i] - kTailBytes);
    const long long k0 = c * kIdat, len = zlen - k0 < kIdat ? zlen - k0 : kIdat;
    uint8_t *chunk = o + kHeadBytes + c * (kIdat + 12);
    if (threadIdx.x == 0) put_be32(chunk, (uint32_t)len);
    __syncthreads();
    const uint32_t *words = ws.words + (long long)i * ws.wcap;
    // "IDAT" + payload as one sequence q = 0 .. 4 + len, PACK_BPT bytes per thread
    uint32_t crc = ~0u;
    const long long q0 = (long long)threadIdx.x * PACK_BPT;
    long long cnt = 0;
    for (int j = 0; j < PACK_BPT; j++) {
        const long long q = q0 + j;
        if (q >= 4 + len) break;
        const uint8_t v = q < 4 ? (uint8_t)"IDAT"[q] : zlib_byte(zh, words, db, adler, k0 + q - 4);
        chunk[4 + q] = v;
        crc = table[(crc ^ v) & 0xFF] ^ (crc >> 8);
        ++cnt;
    }
    scrc[threadIdx.x] = ~crc;
    slen[threadIdx.x] = cnt;
    __syncthreads();
    for (int stride = 1; stride < THREADS; stride <<= 1) {        // combine neighbours, pairs of pieces at a time
        if ((threadIdx.x & (2 * stride - 1)) == 0) {
            const int r = threadIdx.x + stride;
            scrc[threadIdx.x] = crc32_combine(scrc[threadIdx.x], scrc[r], slen[r]);
            slen[threadIdx.x] += slen[r];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) put_be32(chunk + 8 + len, scrc[0]);
}

bool caps_ok(int n_img, int max_h, int max_w) {
    return n_img > 0 && n_img <= 65535 && max_h > 0 && max_w > 0 && max_h <= 65535 && max_w <= 65535 &&
           data_size(max_h, max_w) < (1ll << 30) && (long long)n_img * max_blocks(data_size(max_h, max_w)) < (1ll << 31) &&
           (long long)n_img * ((data_size(max_h, max_w) + TILE - 1) / TILE) < (1ll << 31) &&
           (long long)n_img * num_chunks(zlib_bound(data_size(max_h, max_w))) < (1ll << 31);
}

}  // namespace
}  // namespace pn

using namespace pn;

extern "C" int pn_png_encode_bound(int h, int w, int64_t *bytes_host) {
    PN_CHECK_ARG(bytes_host, "pn_png_encode_bound: null pointer");
    PN_CHECK_ARG(h >= 0 && w >= 0 && h <= 65535 && w <= 65535 && data_size(h, w) < (1ll << 30),
                 "pn_png_encode_bound: bad size %d x %d", h, w);
    *bytes_host = encode_bound(h, w);
    return PN_OK;
}

extern "C" int pn_png_encode_workspace(int n_img, int max_h, int max_w, size_t *bytes_host) {
    PN_CHECK_ARG(bytes_host, "pn_png_encode_workspace: null pointer");
    PN_CHECK_ARG(caps_ok(n_img, max_h, max_w), "pn_png_encode_workspace: bad capacity (%d images, %d x %d)", n_img, max_h, max_w);
    *bytes_host = layout(n_img, max_h, max_w).bytes;
    return PN_OK;
}

extern "C" int pn_png_encode(const uint8_t *frames, int n_img, int max_h, int max_w, int64_t frame_stride, const int *frame_hw,
                             uint8_t *out, int64_t out_capacity, int64_t *out_offsets, void *workspace, size_t ws_bytes,
                             pn_stream_t stream) {
    PN_CHECK_ARG(frames && out && out_offsets && workspace, "pn_png_encode: null pointer");
    PN_CHECK_ARG(caps_ok(n_img, max_h, max_w), "pn_png_encode: bad capacity (%d images, %d x %d)", n_img, max_h, max_w);
    PN_CHECK_ARG(frame_stride >= 3ll * max_h * max_w, "pn_png_encode: frame_stride %lld < 3 * max_h * max_w",
                 (long long)frame_stride);
    PN_CHECK_ARG(((uintptr_t)workspace & 255) == 0, "pn_png_encode: workspace must be 256-byte aligned");
    const Layout L = layout(n_img, max_h, max_w);
    PN_CHECK_ARG(ws_bytes >= L.bytes, "pn_png_encode: workspace %zu < %zu bytes (pn_png_encode_workspace)", ws_bytes, L.bytes);
    const long long bound = encode_bound(max_h, max_w);
    PN_CHECK_ARG(out_capacity / n_img >= bound, "pn_png_encode: out_capacity %lld < %d x %lld bytes (pn_png_encode_bound)",
                 (long long)out_capacity, n_img, bound);
    const Args a{frames, n_img, max_h, max_w, frame_stride, frame_hw, out, out_offsets};
    const Ws w = bind(workspace, L);
    const cudaStream_t st = as_stream(stream);
    const unsigned tiles = (unsigned)(n_img * L.tcap), blocks = (unsigned)(n_img * L.bcap), chunks = (unsigned)(n_img * L.ccap);
    PN_CHECK_CUDA(cudaMemsetAsync(w.adler, 0, 16ull * n_img, st));
    filter_kernel<<<tiles, THREADS, 0, st>>>(a, w);
    PN_CHECK_LAUNCH();
    carry_kernel<<<n_img, CTA_THREADS, 0, st>>>(a, w);
    PN_CHECK_LAUNCH();
    symbols_kernel<false><<<tiles, THREADS, 0, st>>>(a, w);
    PN_CHECK_LAUNCH();
    scan_kernel<<<n_img, CTA_THREADS, 0, st>>>(a, w);
    PN_CHECK_LAUNCH();
    symbols_kernel<true><<<tiles, THREADS, 0, st>>>(a, w);
    PN_CHECK_LAUNCH();
    trees_kernel<<<blocks, THREADS, 0, st>>>(a, w);
    PN_CHECK_LAUNCH();
    place_kernel<<<1, CTA_THREADS, 0, st>>>(a, w);
    PN_CHECK_LAUNCH();
    clear_kernel<<<4 * num_sms(), THREADS, 0, st>>>(a, w);
    PN_CHECK_LAUNCH();
    emit_kernel<<<blocks, THREADS, 0, st>>>(a, w);
    PN_CHECK_LAUNCH();
    pack_kernel<<<chunks, THREADS, 0, st>>>(a, w);
    PN_CHECK_LAUNCH();
    return PN_OK;
}
