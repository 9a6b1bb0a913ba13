// pn_jpeg_encode: uint8 BGR frames on the device -> baseline JPEG files, bit-exact with cv2.imencode(".jpg") (arithmetic:
// jpeg_encode.cuh).
//
// One call encodes a batch in seven launches whose geometry depends only on the capacity (n_img, max_h, max_w, sampling, restart
// interval), so the call can be captured in a CUDA graph; quality, tables and the header template are kernel parameters:
//   transform  eight threads per 8x8 block: colour conversion + downsampling of one row each, jpeg_fdct_islow's row pass, its
//              column pass, quantisation, coefficients stored in zig-zag order.  MCU padding blocks get their DC here: it is the
//              quantised DC (the sum of the samples) of a real block of the same MCU, recomputed rather than waited for
//   length     a thread per block: DC difference (the predictor is a closed-form block index) and the block's Huffman bit length
//   scan       a CTA per image: exclusive sum of the lengths, restart intervals padded to whole bytes, every block's bit position
//              in the image's unstuffed stream; zeroes the words of that stream
//   emit       a thread per block writes its codes at its bit position: words it shares with a neighbour by atomicOr, the others
//              by plain stores; the last block of an interval appends the 1-bit padding
//   count      a CTA per image counts the 0xFF bytes of its stream: the file's size
//   offsets    one CTA: exclusive sum of the sizes into out_offsets
//   pack       a CTA per image: header (height and width patched into SOF0), the stream with 0x00 after every 0xFF, RSTn before
//              every interval but the first, EOI
#include "common.cuh"
#include "jpeg_encode.cuh"

namespace pn {
namespace {

using namespace jpege;

constexpr int THREADS = 256;
constexpr int CTA_THREADS = 1024;                 // the per-image kernels
constexpr int PACK_BYTES = 16;                    // unstuffed bytes per thread and round in pack

struct EncParams {
    Tables T;
    uint8_t header[kMaxHeader];
    int header_len, sof_hw;
};

struct Args {
    const uint8_t *frames;
    int n_img, max_h, max_w;
    int64_t stride;
    const int *frame_hw;
    int sampling, rst;
    uint8_t *out;
    int64_t *offsets;
};

struct Layout {
    size_t coef, len, segbits, segbyte, words, size, bytes;
    long long bcap, scap, wcap;                   // per image: blocks, restart intervals, unstuffed words
};

size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

bool cap_geom(int max_h, int max_w, int sampling, int rst, Geom *g) { return geometry(max_h, max_w, sampling, rst, g); }

Layout layout(int n_img, const Geom &g) {
    Layout L;
    L.bcap = g.nblk;
    L.scap = g.nseg;
    L.wcap = (g.nblk * kMaxBlockBits / 8 + g.nseg + 8) / 4 + 1;
    size_t o = 0;
    auto take = [&](size_t bytes) { const size_t at = o; o = align256(o + bytes); return at; };
    L.coef = take(128ull * n_img * L.bcap);
    L.len = take(4ull * n_img * L.bcap);
    L.segbits = take(4ull * n_img * L.scap);
    L.segbyte = take(4ull * n_img * (L.scap + 1));
    L.words = take(4ull * n_img * L.wcap);
    L.size = take(8ull * n_img);
    L.bytes = o;
    return L;
}

struct Ws {
    int16_t *coef;
    uint32_t *len;        // block bit length (length), then bit position in the image's unstuffed stream (scan)
    uint32_t *segbits;    // exclusive bit sum at each interval's first block
    uint32_t *segbyte;    // each interval's first byte in the unstuffed stream; [nseg]: the stream's length
    uint32_t *words;      // unstuffed streams, big-endian bit order within a word
    long long *size;      // file sizes
    long long bcap, scap, wcap;
};

Ws bind(void *base, const Layout &L) {
    char *b = static_cast<char *>(base);
    return Ws{reinterpret_cast<int16_t *>(b + L.coef), reinterpret_cast<uint32_t *>(b + L.len),
              reinterpret_cast<uint32_t *>(b + L.segbits), reinterpret_cast<uint32_t *>(b + L.segbyte),
              reinterpret_cast<uint32_t *>(b + L.words), reinterpret_cast<long long *>(b + L.size), L.bcap, L.scap, L.wcap};
}

// Image i's geometry: its own size with frame_hw (a size outside 1..max is an empty file), else max_h x max_w.
__device__ __forceinline__ Geom image_geom(const Args &a, int i) {
    int h = a.max_h, w = a.max_w;
    if (a.frame_hw) {
        h = a.frame_hw[2 * i];
        w = a.frame_hw[2 * i + 1];
        if (h < 1 || w < 1 || h > a.max_h || w > a.max_w) h = w = 0;
    }
    Geom g;
    geometry(h, w, a.sampling, a.rst, &g);
    return g;
}

__device__ __forceinline__ long long seg_blocks(const Geom &g) { return g.rst > 0 ? (long long)g.rst * g.bpm : g.nblk; }

// ---- transform: eight threads per block ----------------------------------------------------------------------------------------
__global__ void __launch_bounds__(THREADS) transform_kernel(Args a, Ws ws, const __grid_constant__ EncParams p) {
    __shared__ Recip sq[2][64];
    __shared__ int sd[THREADS / 8][64];
    for (int k = threadIdx.x; k < 128; k += THREADS) sq[k >> 6][k & 63] = p.T.quant[k >> 6][k & 63];
    __syncthreads();
    const int grp = threadIdx.x >> 3, r = threadIdx.x & 7;
    const long long total = (long long)a.n_img * ws.bcap;
    for (long long g0 = blockIdx.x * (long long)(THREADS / 8); g0 < total; g0 += (long long)gridDim.x * (THREADS / 8)) {
        const long long gb = g0 + grp;
        const int i = gb < total ? (int)(gb / ws.bcap) : 0;
        const long long blk = gb - (long long)i * ws.bcap;
        Geom g = image_geom(a, i);
        const bool live = gb < total && blk < g.nblk;
        int c = 0, bx = 0, by = 0, mx = 0, sx = 0, sy = 0;
        bool dummy = false;
        const uint8_t *frame = a.frames + (long long)i * a.stride;
        if (live) {
            block_place(g, blk, &c, &bx, &by, &mx);
            dummy = dummy_source(g, c, bx, by, mx, &sx, &sy);
        }
        int16_t *zz = ws.coef + gb * 64;
        if (live && !dummy) {
            int *d = sd[grp] + 8 * r;
#pragma unroll 1
            for (int x = 0; x < 8; ++x) d[x] = sample(g, frame, c, bx * 8 + x, by * 8 + r) - 128;
            fdct_pass(d, 1, 0);
        }
        __syncwarp();
        if (live && !dummy) {
            int *d = sd[grp] + r;
            fdct_pass(d, 8, 1);
#pragma unroll
            for (int y = 0; y < 8; ++y) zz[zigzag_of(y * 8 + r)] = (int16_t)quantize(d[8 * y], sq[c ? 1 : 0][y * 8 + r]);
        }
        // padding block: the quantised DC of its source block (the DCT's DC output is the sum of the samples)
        int sum = 0;
        if (live && dummy) {
#pragma unroll 1
            for (int x = 0; x < 8; ++x) sum += sample(g, frame, c, sx * 8 + x, sy * 8 + r) - 128;
        }
        sum += __shfl_xor_sync(0xffffffffu, sum, 1);
        sum += __shfl_xor_sync(0xffffffffu, sum, 2);
        sum += __shfl_xor_sync(0xffffffffu, sum, 4);
        if (live && dummy) {
#pragma unroll
            for (int k = 0; k < 8; ++k) zz[8 * r + k] = 0;
            if (r == 0) zz[0] = (int16_t)quantize(sum, sq[c ? 1 : 0][0]);
        }
        __syncwarp();
    }
}

__device__ __forceinline__ void load_huff(const EncParams &p, HuffEnc *sh) {
    const uint32_t *src = reinterpret_cast<const uint32_t *>(&p.T.dc[0]);
    uint32_t *dst = reinterpret_cast<uint32_t *>(sh);
    static_assert(sizeof(HuffEnc) % 4 == 0, "HuffEnc is copied as words");
    for (int k = threadIdx.x; k < (int)(4 * sizeof(HuffEnc) / 4); k += blockDim.x) dst[k] = src[k];
    __syncthreads();
}

// ---- length: a thread per block ----------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(THREADS) length_kernel(Args a, Ws ws, const __grid_constant__ EncParams p) {
    __shared__ HuffEnc sh[4];                     // dc0, dc1, ac0, ac1 (Tables order)
    load_huff(p, sh);
    const long long total = (long long)a.n_img * ws.bcap;
    for (long long gb = blockIdx.x * (long long)THREADS + threadIdx.x; gb < total; gb += (long long)gridDim.x * THREADS) {
        const int i = (int)(gb / ws.bcap);
        const long long blk = gb - (long long)i * ws.bcap;
        const Geom g = image_geom(a, i);
        if (blk >= g.nblk) continue;
        int c, bx, by, mx;
        block_place(g, blk, &c, &bx, &by, &mx);
        const int16_t *zz = ws.coef + gb * 64;
        const long long pb = dc_pred_block(g, blk);
        const int diff = zz[0] - (pb >= 0 ? ws.coef[(gb - blk + pb) * 64] : 0);
        CountBits cb;
        encode_block(zz, diff, sh[c ? 1 : 0], sh[2 + (c ? 1 : 0)], cb);
        ws.len[gb] = cb.bits;
    }
}

// ---- per-image CTA helpers -----------------------------------------------------------------------------------------------------
template <typename T>
__device__ T cta_exclusive_scan(T v, T *total, T *sm) {   // sm: CTA_THREADS / 32 + 1 entries
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    T x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const T y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) sm[warp] = x;
    __syncthreads();
    if (warp == 0) {
        const T t = lane < CTA_THREADS / 32 ? sm[lane] : T(0);
        T s = t;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const T y = __shfl_up_sync(0xffffffffu, s, o);
            if (lane >= o) s += y;
        }
        if (lane < CTA_THREADS / 32) sm[lane] = s - t;
        if (lane == 31) sm[CTA_THREADS / 32] = s;
    }
    __syncthreads();
    const T r = sm[warp] + x - v;
    *total = sm[CTA_THREADS / 32];
    __syncthreads();
    return r;
}

// ---- scan: a CTA per image -------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(CTA_THREADS) scan_kernel(Args a, Ws ws) {
    __shared__ uint32_t sm[CTA_THREADS / 32 + 1];
    __shared__ uint32_t s_run;
    const int i = blockIdx.x;
    const Geom g = image_geom(a, i);
    uint32_t *len = ws.len + (long long)i * ws.bcap;
    uint32_t *segbits = ws.segbits + (long long)i * ws.scap, *segbyte = ws.segbyte + (long long)i * (ws.scap + 1);
    if (threadIdx.x == 0) s_run = 0;
    __syncthreads();
    // bits before each block, over the whole image
    for (long long b0 = 0; b0 < g.nblk; b0 += CTA_THREADS) {
        const long long b = b0 + threadIdx.x;
        const uint32_t v = b < g.nblk ? len[b] : 0u;
        uint32_t tot;
        const uint32_t e = cta_exclusive_scan<uint32_t>(v, &tot, sm) + s_run;
        if (b < g.nblk) len[b] = e;
        __syncthreads();
        if (threadIdx.x == 0) s_run += tot;
        __syncthreads();
    }
    const uint32_t total_bits = s_run;
    __syncthreads();
    if (threadIdx.x == 0) s_run = 0;
    __syncthreads();
    // restart intervals: first bit, whole bytes
    const long long per = seg_blocks(g);
    for (int s0 = 0; s0 < g.nseg; s0 += CTA_THREADS) {
        const int s = s0 + threadIdx.x;
        uint32_t bytes = 0;
        if (s < g.nseg) {
            const long long b = (long long)s * per, e = b + per < g.nblk ? b + per : g.nblk;
            const uint32_t first = len[b], last = e < g.nblk ? len[e] : total_bits;
            segbits[s] = first;
            bytes = (last - first + 7) / 8;
        }
        uint32_t tot;
        const uint32_t o = cta_exclusive_scan<uint32_t>(bytes, &tot, sm) + s_run;
        if (s < g.nseg) segbyte[s] = o;
        __syncthreads();
        if (threadIdx.x == 0) s_run += tot;
        __syncthreads();
    }
    const uint32_t ubytes = s_run;
    if (threadIdx.x == 0) segbyte[g.nseg] = ubytes;
    // bit positions in the unstuffed stream
    for (long long b = threadIdx.x; b < g.nblk; b += CTA_THREADS) {
        const int s = (int)(b / per);
        len[b] = 8u * segbyte[s] + (len[b] - segbits[s]);
    }
    uint32_t *words = ws.words + (long long)i * ws.wcap;
    for (long long k = threadIdx.x; k < (ubytes + 3) / 4; k += CTA_THREADS) words[k] = 0;
}

// ---- emit: a thread per block --------------------------------------------------------------------------------------------------------
struct WordSink {
    uint32_t *words;
    uint32_t wi, cur;
    int fill;
    bool first;
    __device__ __forceinline__ void store() {
        if (first) atomicOr(words + wi, cur);
        else words[wi] = cur;
        first = false;
    }
    __device__ __forceinline__ void operator()(uint32_t code, int size) {
        while (size > 0) {
            const int take = size < 32 - fill ? size : 32 - fill;
            const uint32_t part = (code >> (size - take)) & (take == 32 ? ~0u : ((1u << take) - 1u));
            cur |= part << (32 - fill - take);
            fill += take;
            size -= take;
            if (fill == 32) {
                store();
                ++wi;
                cur = 0;
                fill = 0;
            }
        }
    }
    __device__ __forceinline__ void finish() {
        if (fill) atomicOr(words + wi, cur);   // shared with the next block
    }
};

__global__ void __launch_bounds__(THREADS) emit_kernel(Args a, Ws ws, const __grid_constant__ EncParams p) {
    __shared__ HuffEnc sh[4];
    load_huff(p, sh);
    const long long total = (long long)a.n_img * ws.bcap;
    for (long long gb = blockIdx.x * (long long)THREADS + threadIdx.x; gb < total; gb += (long long)gridDim.x * THREADS) {
        const int i = (int)(gb / ws.bcap);
        const long long blk = gb - (long long)i * ws.bcap;
        const Geom g = image_geom(a, i);
        if (blk >= g.nblk) continue;
        int c, bx, by, mx;
        block_place(g, blk, &c, &bx, &by, &mx);
        const int16_t *zz = ws.coef + gb * 64;
        const long long pb = dc_pred_block(g, blk);
        const int diff = zz[0] - (pb >= 0 ? ws.coef[(gb - blk + pb) * 64] : 0);
        const uint32_t pos = ws.len[gb];
        WordSink sink{ws.words + (long long)i * ws.wcap, pos >> 5, 0u, (int)(pos & 31), true};
        encode_block(zz, diff, sh[c ? 1 : 0], sh[2 + (c ? 1 : 0)], sink);
        if ((blk + 1) % seg_blocks(g) == 0 || blk + 1 == g.nblk) {       // end of a restart interval: pad with 1-bits
            const int used = (sink.fill & 7);
            if (used) sink((1u << (8 - used)) - 1u, 8 - used);
        }
        sink.finish();
    }
}

__device__ __forceinline__ uint32_t ubyte(const uint32_t *words, uint32_t k) { return (words[k >> 2] >> (24 - 8 * (k & 3))) & 0xFFu; }

// ---- count: a CTA per image ------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(CTA_THREADS) count_kernel(Args a, Ws ws, const __grid_constant__ EncParams p) {
    __shared__ uint32_t s_ff;
    const int i = blockIdx.x;
    const Geom g = image_geom(a, i);
    if (threadIdx.x == 0) s_ff = 0;
    __syncthreads();
    const uint32_t *words = ws.words + (long long)i * ws.wcap;
    const uint32_t ubytes = g.nblk ? ws.segbyte[(long long)i * (ws.scap + 1) + g.nseg] : 0u;
    uint32_t ff = 0;
    for (uint32_t k = threadIdx.x; k < ubytes; k += CTA_THREADS) ff += ubyte(words, k) == 0xFFu;
    ff = __reduce_add_sync(0xffffffffu, ff);
    if ((threadIdx.x & 31) == 0 && ff) atomicAdd(&s_ff, ff);
    __syncthreads();
    if (threadIdx.x == 0)
        ws.size[i] = g.nblk ? (long long)p.header_len + ubytes + s_ff + 2ll * (g.nseg - 1) + 2 : 0;
}

// ---- offsets: one CTA ----------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(CTA_THREADS) offsets_kernel(Args a, Ws ws) {
    __shared__ long long sm[CTA_THREADS / 32 + 1];
    long long run = 0;
    for (int i0 = 0; i0 < a.n_img; i0 += CTA_THREADS) {
        const int i = i0 + threadIdx.x;
        long long tot;
        const long long o = cta_exclusive_scan<long long>(i < a.n_img ? ws.size[i] : 0, &tot, sm) + run;
        if (i < a.n_img) a.offsets[i] = o;
        run += tot;
    }
    if (threadIdx.x == 0) a.offsets[a.n_img] = run;
}

// ---- pack: a CTA per image ------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(CTA_THREADS) pack_kernel(Args a, Ws ws, const __grid_constant__ EncParams p) {
    __shared__ uint32_t sm[CTA_THREADS / 32 + 1];
    __shared__ uint32_t s_run;
    const int i = blockIdx.x;
    const Geom g = image_geom(a, i);
    if (!g.nblk) return;
    uint8_t *o = a.out + a.offsets[i];
    const long long size = ws.size[i];
    for (int t = threadIdx.x; t < p.header_len; t += CTA_THREADS) {
        uint8_t v = p.header[t];
        if (t == p.sof_hw) v = (uint8_t)(g.h >> 8);
        else if (t == p.sof_hw + 1) v = (uint8_t)g.h;
        else if (t == p.sof_hw + 2) v = (uint8_t)(g.w >> 8);
        else if (t == p.sof_hw + 3) v = (uint8_t)g.w;
        o[t] = v;
    }
    if (threadIdx.x == 0) {
        o[size - 2] = 0xFF;
        o[size - 1] = 0xD9;
        s_run = 0;
    }
    __syncthreads();
    const uint32_t *words = ws.words + (long long)i * ws.wcap;
    const uint32_t *segbyte = ws.segbyte + (long long)i * (ws.scap + 1);
    const uint32_t ubytes = segbyte[g.nseg];
    uint8_t *data = o + p.header_len;
    for (uint32_t c0 = 0; c0 < ubytes; c0 += CTA_THREADS * PACK_BYTES) {
        const uint32_t k0 = c0 + threadIdx.x * PACK_BYTES;
        uint32_t ff = 0;
#pragma unroll
        for (int j = 0; j < PACK_BYTES; ++j) ff += k0 + j < ubytes && ubyte(words, k0 + j) == 0xFFu;
        uint32_t tot;
        uint32_t before = cta_exclusive_scan<uint32_t>(ff, &tot, sm) + s_run;
        if (k0 < ubytes) {
            int lo = 0, hi = g.nseg - 1;                                   // the interval holding byte k0
            while (lo < hi) {
                const int mid = (lo + hi + 1) >> 1;
                if (segbyte[mid] <= k0) lo = mid; else hi = mid - 1;
            }
            int s = lo;
            for (int j = 0; j < PACK_BYTES && k0 + j < ubytes; ++j) {
                const uint32_t k = k0 + j;
                while (s + 1 < g.nseg && segbyte[s + 1] <= k) ++s;
                const long long at = (long long)k + before + 2ll * s;
                if (s > 0 && k == segbyte[s]) {
                    data[at - 2] = 0xFF;
                    data[at - 1] = (uint8_t)(0xD0 + ((s - 1) & 7));
                }
                const uint32_t b = ubyte(words, k);
                data[at] = (uint8_t)b;
                if (b == 0xFFu) {
                    data[at + 1] = 0;
                    ++before;
                }
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) s_run += tot;
        __syncthreads();
    }
}

bool caps_ok(int n_img, int max_h, int max_w, int sampling, int rst, Geom *g) {
    return n_img > 0 && n_img <= 65535 && max_h > 0 && max_w > 0 && max_h <= 65500 && max_w <= 65500 && rst >= 0 &&
           rst <= 65535 && cap_geom(max_h, max_w, sampling, rst, g) &&
           g->nblk * (long long)kMaxBlockBits + 8ll * g->nseg + 64 < (1ll << 32);
}

int header_of(const Tables &T, int sampling, int rst, uint8_t *hdr, int *sof) { return write_header(T, sampling, rst, 0, 0, hdr, sof); }

}  // namespace
}  // namespace pn

using namespace pn;

extern "C" int pn_jpeg_encode_bound(int h, int w, int sampling, int restart_interval, int64_t *bytes_host) {
    PN_CHECK_ARG(bytes_host, "pn_jpeg_encode_bound: null pointer");
    Geom g;
    PN_CHECK_ARG(h >= 0 && w >= 0 && h <= 65500 && w <= 65500 && restart_interval >= 0 && restart_interval <= 65535 &&
                     geometry(h, w, sampling, restart_interval, &g),
                 "pn_jpeg_encode_bound: bad arguments (%d x %d, sampling 0x%x, restart interval %d)", h, w, sampling,
                 restart_interval);
    Tables T;
    make_tables(95, &T);
    uint8_t hdr[kMaxHeader];
    int sof;
    *bytes_host = encode_bound(g, header_of(T, sampling, restart_interval, hdr, &sof));
    return PN_OK;
}

extern "C" int pn_jpeg_encode_workspace(int n_img, int max_h, int max_w, int sampling, int restart_interval, size_t *bytes_host) {
    PN_CHECK_ARG(bytes_host, "pn_jpeg_encode_workspace: null pointer");
    Geom g;
    PN_CHECK_ARG(caps_ok(n_img, max_h, max_w, sampling, restart_interval, &g),
                 "pn_jpeg_encode_workspace: bad capacity (%d images, %d x %d, sampling 0x%x, restart interval %d)", n_img, max_h,
                 max_w, sampling, restart_interval);
    *bytes_host = layout(n_img, g).bytes;
    return PN_OK;
}

extern "C" int pn_jpeg_encode(const uint8_t *frames, int n_img, int max_h, int max_w, int64_t frame_stride, const int *frame_hw,
                              int quality, int sampling, int restart_interval, uint8_t *out, int64_t out_capacity,
                              int64_t *out_offsets, void *workspace, size_t ws_bytes, pn_stream_t stream) {
    PN_CHECK_ARG(frames && out && out_offsets && workspace, "pn_jpeg_encode: null pointer");
    Geom g;
    PN_CHECK_ARG(caps_ok(n_img, max_h, max_w, sampling, restart_interval, &g),
                 "pn_jpeg_encode: bad capacity (%d images, %d x %d, sampling 0x%x, restart interval %d)", n_img, max_h, max_w,
                 sampling, restart_interval);
    PN_CHECK_ARG(quality >= 0 && quality <= 100, "pn_jpeg_encode: quality %d outside 0..100", quality);
    PN_CHECK_ARG(frame_stride >= 3ll * max_h * max_w, "pn_jpeg_encode: frame_stride %lld < 3 * max_h * max_w",
                 (long long)frame_stride);
    PN_CHECK_ARG(((uintptr_t)workspace & 255) == 0, "pn_jpeg_encode: workspace must be 256-byte aligned");
    const Layout L = layout(n_img, g);
    PN_CHECK_ARG(ws_bytes >= L.bytes, "pn_jpeg_encode: workspace %zu < %zu bytes (pn_jpeg_encode_workspace)", ws_bytes, L.bytes);
    EncParams p;
    memset(&p, 0, sizeof(p));
    make_tables(quality, &p.T);
    p.header_len = header_of(p.T, sampling, restart_interval, p.header, &p.sof_hw);
    const long long bound = encode_bound(g, p.header_len);
    PN_CHECK_ARG(out_capacity / n_img >= bound, "pn_jpeg_encode: out_capacity %lld < %d x %lld bytes (pn_jpeg_encode_bound)",
                 (long long)out_capacity, n_img, bound);
    const Args a{frames, n_img, max_h, max_w, frame_stride, frame_hw, sampling, restart_interval, out, out_offsets};
    const Ws w = bind(workspace, L);
    const cudaStream_t st = as_stream(stream);
    const int grid = 4 * num_sms();
    transform_kernel<<<grid, THREADS, 0, st>>>(a, w, p);
    PN_CHECK_LAUNCH();
    length_kernel<<<grid, THREADS, 0, st>>>(a, w, p);
    PN_CHECK_LAUNCH();
    scan_kernel<<<n_img, CTA_THREADS, 0, st>>>(a, w);
    PN_CHECK_LAUNCH();
    emit_kernel<<<grid, THREADS, 0, st>>>(a, w, p);
    PN_CHECK_LAUNCH();
    count_kernel<<<n_img, CTA_THREADS, 0, st>>>(a, w, p);
    PN_CHECK_LAUNCH();
    offsets_kernel<<<1, CTA_THREADS, 0, st>>>(a, w);
    PN_CHECK_LAUNCH();
    pack_kernel<<<n_img, CTA_THREADS, 0, st>>>(a, w, p);
    PN_CHECK_LAUNCH();
    return PN_OK;
}
