// B3, stand-alone, stride 1 (dilation 1 or 2), bf16 -- the depthwise 3x3 + bias + ReLU6 of the blocks that are not fused with
// their pointwise conv (posenet/models/mobilenet_v1.py:60-62,66; at C2: blocks 12 and 13, 512 / 1024 channels at 33 x 33), as
// warp-autonomous pipelines (the design of sepwarp.cu without the tensor phase):
//   * a work item is a column strip of 4 output pixels x 64 channels x a run of output rows of ONE residue class mod the
//     dilation (rows c, c + D, c + 2D, ...: in that row space the dilated stencil is dense again, so the 3-row window slides
//     with one new row per output row); the TMA tensor map traverses the row dimension with element stride D, so the rows of
//     the class arrive densely packed;
//   * lane l owns the channel pair (2l, 2l + 1): 4 bytes of every pixel, one conflict-free 128 B wavefront per warp load,
//     the window as fp32 pairs in registers, 36 packed FFMA2 per output row, results stored as 128 B coalesced pixel rows;
//   * lane 0 streams the strip through a private two-stage TMA ring (OOB zero fill == zero padding); no CTA-wide barrier.
// ~11 thread-instructions per output element against ~23 for the tile kernel in dwconv.cu (which reloads the window for
// every output row and its weights for every strip); that kernel remains for fp32, stride 2 and dilation 4.
#include <cuda.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "common.cuh"
#include "ptx.cuh"

namespace pn {

// rows (of one class) per TMA chunk / chunks in flight per warp / warps per CTA, per dilation (measured: dilation 1 prefers
// two 8-row chunks, dilation 2 -- wider patches, more registers -- three 4-row chunks; both 16 warps)
__host__ __device__ constexpr int dww_rows(int d) { return d == 1 ? 8 : 4; }
__host__ __device__ constexpr int dww_stages(int d) { return d == 1 ? 2 : 3; }
constexpr int DWW_PIX = 128;                              // bytes per patch pixel: 64 channels bf16
__host__ __device__ constexpr int dww_ncols(int d) { return 4 + 2 * d; }
__host__ __device__ constexpr int dww_chunk(int d) { return dww_rows(d) * dww_ncols(d) * DWW_PIX; }
__host__ __device__ constexpr int dww_warp_smem(int d) { return dww_stages(d) * dww_chunk(d) + 128; }
__host__ __device__ constexpr int dww_warps(int d) { return 16; }
__host__ __device__ constexpr int dww_smem(int d) { return dww_warps(d) * dww_warp_smem(d) + 1024; }

struct DwwGeom {
    int n, h, w, c;
    int cblocks, strips, nq, rb;   // 64-channel blocks, 4-pixel column strips, row blocks per class, class rows per block
    int items;                     // n * nq * D * strips * cblocks (< 2^31: 32-bit index arithmetic in the kernel)
};

__device__ __forceinline__ void dww_stg_u32_if(void *p, uint32_t v, bool on) {          // one predicated STG, no branch
    if (on) asm volatile("st.global.b32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t dww_lds_u32(uint32_t addr) {
    uint32_t r;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(r) : "r"(addr));
    return r;
}

template <int D>
__global__ void __launch_bounds__(dww_warps(D) * 32, 1)
dwwarp_kernel(const __grid_constant__ CUtensorMap tmap_x, const float *__restrict__ dw_w, const float *__restrict__ dw_b,
              __nv_bfloat16 *__restrict__ y, const DwwGeom g) {
    constexpr int NCOLS = dww_ncols(D), CHUNK = dww_chunk(D), WARPS = dww_warps(D), DWW_ROWS = dww_rows(D), DWW_STAGES = dww_stages(D);
    extern __shared__ uint8_t dww_raw[];
    const uint32_t base = (smem_u32(dww_raw) + 1023u) & ~1023u;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t sRing = base + (uint32_t)warp * dww_warp_smem(D), bars = sRing + DWW_STAGES * CHUNK;
    if (lane == 0) {
        for (int s_ = 0; s_ < DWW_STAGES; ++s_) mbar_init(bars + 8u * s_, 1);
        mbar_fence_init();
        if (warp == 0) tma_prefetch_desc(&tmap_x);
    }
    pdl_launch_dependents();
    __syncthreads();
    pdl_wait();

    auto unpack = [](uint32_t r) { return make_float2(__uint_as_float(r << 16), __uint_as_float(r & 0xffff0000u)); };
    uint32_t phase_bits = 0;
    const int total_warps = (int)gridDim.x * WARPS, first_item = (int)blockIdx.x * WARPS + warp;

    // item -> (image, row block, class, strip, channel block); channel blocks fastest: neighbouring warps read the same pixels
    struct Item { int cb, xs, cls, img, i0, rows_out, nchunks; };
    auto decode = [&](int it) {
        Item t;
        int r_ = it;
        t.cb = (int)(r_ % g.cblocks); r_ /= g.cblocks;
        t.xs = (int)(r_ % g.strips); r_ /= g.strips;
        t.cls = (int)(r_ % D); r_ /= D;
        const int q = (int)(r_ % g.nq);
        t.img = (int)(r_ / g.nq);
        const int rows_c = (g.h - t.cls + D - 1) / D;                    // output rows of this class
        t.i0 = q * g.rb;                                                 // first class row of the block
        t.rows_out = min(g.rb, rows_c - t.i0);
        t.nchunks = t.rows_out > 0 ? (t.rows_out + 2 + DWW_ROWS - 1) / DWW_ROWS : 0;
        return t;
    };
    // Lane 0 runs a producer cursor two chunks ahead of the consumer, across item boundaries: the ring never drains
    // between items, so the first chunk of an item is (normally) already in flight when the previous item ends.
    int p_item = first_item;
    int p_ci = 0;
    uint32_t p_stage = 0;                                                // ring stage of the next chunk to issue
    Item pit = p_item < g.items ? decode(p_item) : Item{0, 0, 0, 0, 0, 0, 0};
    auto issue_next = [&]() {                                            // lane 0: the next chunk in (item, chunk) order, if any
        while (p_item < g.items && p_ci >= pit.nchunks) {                // (skips empty row blocks)
            p_item += total_warps;
            p_ci = 0;
            if (p_item < g.items) pit = decode(p_item);
        }
        if (p_item >= g.items) return;
        const uint32_t s_ = p_stage;
        mbar_expect_tx(bars + 8u * s_, CHUNK);
        tma_load_4d(sRing + s_ * CHUNK, &tmap_x, bars + 8u * s_, pit.cb * 64, pit.xs * 4 - D, pit.cls + D * (pit.i0 - 1 + p_ci * DWW_ROWS), pit.img);
        if (++p_stage == DWW_STAGES) p_stage = 0;
        ++p_ci;
    };
    if (lane == 0)
        for (int s_ = 0; s_ < DWW_STAGES; ++s_) issue_next();
    uint32_t c_stage = 0;                                                // ring stage of the chunk the consumer enters next

    for (int item = first_item; item < g.items; item += total_warps) {
        const Item it = decode(item);
        const int cb = it.cb, cls = it.cls, img = it.img, i0 = it.i0, rows_out = it.rows_out;
        if (rows_out <= 0) continue;
        const int rows_in = rows_out + 2;
        const int x0 = it.xs * 4, ch0 = cb * 64 + 2 * lane;
        const bool ch_ok = ch0 < g.c;                                    // c is a multiple of 8: the pair is in or out as a whole
        float2 wk[9], bias2;
#pragma unroll
        for (int t = 0; t < 9; ++t) wk[t] = ch_ok ? __ldg(reinterpret_cast<const float2 *>(dw_w + (size_t)t * g.c + ch0)) : make_float2(0.f, 0.f);
        bias2 = ch_ok ? __ldg(reinterpret_cast<const float2 *>(dw_b + ch0)) : make_float2(0.f, 0.f);
        // output addressing: one 64-bit row pointer advanced per output row, the strip's pixels one channel row apart
        const size_t pix_bytes = (size_t)g.c * 2, row_bytes = (size_t)D * g.w * pix_bytes;
        char *o_row = reinterpret_cast<char *>(y) + ((((size_t)img * g.h + (cls + D * i0)) * g.w + x0) * g.c + ch0) * 2;
        bool okp[4];
#pragma unroll
        for (int p = 0; p < 4; ++p) okp[p] = ch_ok && x0 + p < g.w;
        float2 ring[3][NCOLS];
        uint32_t stage_addr = 0;
#pragma unroll 1
        for (int r0 = 0; r0 < rows_in; r0 += 3) {
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                const int r = r0 + j;
                if (r >= rows_in) break;
                const int rr = r & (DWW_ROWS - 1);
                if (rr == 0) {                                            // entering a new chunk: wait for its bytes
                    const uint32_t s = c_stage;
                    mbar_wait(bars + 8u * s, (phase_bits >> s) & 1u);
                    phase_bits ^= 1u << s;
                    stage_addr = sRing + s * CHUNK + (uint32_t)lane * 4u;
                    if (++c_stage == DWW_STAGES) c_stage = 0;
                }
                {
                    const uint32_t rp = stage_addr + (uint32_t)rr * (NCOLS * DWW_PIX);
#pragma unroll
                    for (int c = 0; c < NCOLS; ++c) ring[j][c] = unpack(dww_lds_u32(rp + (uint32_t)c * DWW_PIX));
                }
                const bool refill = (rr == DWW_ROWS - 1 || r == rows_in - 1);
                if (r >= 2) {
                    float2 acc[4] = {bias2, bias2, bias2, bias2};
#pragma unroll
                    for (int ky = 0; ky < 3; ++ky) {
                        const int slot = (j + 1 + ky) % 3;                // class rows r-2, r-1, r
#pragma unroll
                        for (int c = 0; c < NCOLS; ++c)
#pragma unroll
                            for (int p = 0; p < 4; ++p)
#pragma unroll
                                for (int kx = 0; kx < 3; ++kx)
                                    if (p + kx * D == c) acc[p] = ffma2(ring[slot][c], wk[ky * 3 + kx], acc[p]);
                    }
                    char *o = o_row;
#pragma unroll
                    for (int p = 0; p < 4; ++p) {
                        dww_stg_u32_if(o, relu6_bf16x2(acc[p]), okp[p]);
                        o += pix_bytes;
                    }
                    o_row += row_bytes;
                }
                if (refill) {                                             // every lane has consumed the chunk's last row: its stage
                    __syncwarp();                                         // takes the chunk two ahead (of this item or the next)
                    if (lane == 0) issue_next();
                }
            }
        }
    }
}

// ---- host side ---------------------------------------------------------------------------------------------
bool dwwarp_supported(int c, int stride, int dil, int dtype) {
    return dtype == PN_BF16 && stride == 1 && (dil == 1 || dil == 2) && c % 8 == 0;
}

int dwwarp_prepare(DwWarpOp *op, const void *x, int n, int h, int wd, int c, int dil) {
    PN_CHECK_ARG(x && n > 0 && h > 0 && wd > 0 && dwwarp_supported(c, 1, dil, PN_BF16), "pn_dwconv3x3: bad shape for the strip kernel");
    memset(op, 0, sizeof(*op));
    DwwGeom g;
    memset(&g, 0, sizeof(g));
    g.n = n; g.h = h; g.w = wd; g.c = c;
    g.cblocks = ceil_div(c, 64);
    g.strips = ceil_div(wd, 4);
    const int rows_c = ceil_div(h, dil);                                  // rows of the largest class
    const long long warps = (long long)num_sms() * dww_warps(dil);
    const long long per_q = (long long)n * dil * g.strips * g.cblocks;
    const int max_nq = ceil_div(rows_c, 8);                               // row blocks of at least 8 rows
    long long nq = 1;
    // as in sepwarp.cu: items go to the warps round-robin (channel blocks fastest), so the row-block count is the one that
    // leaves the busiest warp the fewest input rows in a simulation of that assignment
    std::vector<long long> load((size_t)warps);
    long long best = -1;
    for (int cand = 1; cand <= max_nq; ++cand) {
        const int rb = ceil_div(rows_c, cand);
        if (ceil_div(rows_c, rb) != cand) continue;
        const long long items_c = per_q * cand;
        if (items_c > (1ll << 22)) break;
        std::fill(load.begin(), load.end(), 0ll);
        const long long per_cls = (long long)g.strips * g.cblocks;        // items per (image, row block, class)
        long long it = 0;
        int wi = 0;
        for (int img = 0; img < n; ++img)
            for (int q = 0; q < cand; ++q)
                for (int cls = 0; cls < dil; ++cls) {
                    const int rows_cls = (h - cls + dil - 1) / dil, rows_out = rows_cls - q * rb < rb ? rows_cls - q * rb : rb;
                    const long long cost = rows_out > 0 ? rows_out + 2 : 0;
                    for (long long j = 0; j < per_cls; ++j, ++it) {
                        load[(size_t)wi] += cost;
                        if (++wi == (int)warps) wi = 0;
                    }
                }
        const long long worst = *std::max_element(load.begin(), load.end());
        if (best < 0 || worst < best) { best = worst; nq = cand; }
    }
    g.rb = ceil_div(rows_c, (int)nq);
    g.nq = ceil_div(rows_c, g.rb);
    const long long items = (long long)n * g.nq * dil * g.strips * g.cblocks;
    PN_CHECK_ARG(items + (long long)num_sms() * 16 < (1ll << 31), "pn_dwconv3x3: problem too large for one launch");
    g.items = (int)items;
    op->dil = dil;
    static_assert(sizeof(DwwGeom) <= sizeof(op->geom), "DwWarpOp::geom too small");
    memcpy(op->geom, &g, sizeof(g));
    const uint64_t dims[4] = {(uint64_t)c, (uint64_t)wd, (uint64_t)h, (uint64_t)n};
    const uint64_t strides[3] = {(uint64_t)c * 2, (uint64_t)wd * c * 2, (uint64_t)h * wd * c * 2};
    const uint32_t box[4] = {64u, (uint32_t)dww_ncols(dil), (uint32_t)(dww_rows(dil) * dil), 1u};   // every dil-th row: dww_rows land
    const uint32_t estr[4] = {1u, 1u, (uint32_t)dil, 1u};
    return encode_tmap(op->tmap_x, x, 2, 4, dims, strides, box, 0, estr);
}

template <int D>
static int dwwarp_launch_t(const DwWarpOp *op, const DwwGeom &g, const float *w, const float *b, void *y, cudaStream_t st) {
    static DeviceOnce once;
    const int dev = current_device();
    auto kern = dwwarp_kernel<D>;
    if (!once.get(dev)) {
        PN_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, dww_smem(D)));
        once.set(dev, 1);
    }
    const long long ctas = ((long long)g.items + dww_warps(D) - 1) / dww_warps(D);
    const int grid = (int)(ctas < num_sms() ? ctas : num_sms());
    PN_CHECK_CUDA(launch_pdl(kern, dim3(grid), dim3(dww_warps(D) * 32), (size_t)dww_smem(D), st, *reinterpret_cast<const CUtensorMap *>(op->tmap_x), w,
                             b, (__nv_bfloat16 *)y, g));
    return PN_OK;
}

int dwwarp_launch(const DwWarpOp *op, const float *w, const float *b, void *y, cudaStream_t st) {
    PN_CHECK_ARG(op && w && b && y, "pn_dwconv3x3: null pointer");
    PN_CHECK_ARG(((uintptr_t)y & 3) == 0 && ((uintptr_t)w & 7) == 0 && ((uintptr_t)b & 7) == 0, "pn_dwconv3x3: misaligned pointer");
    DwwGeom g;
    memcpy(&g, op->geom, sizeof(g));
    return op->dil == 1 ? dwwarp_launch_t<1>(op, g, w, b, y, st) : dwwarp_launch_t<2>(op, g, w, b, y, st);
}

}  // namespace pn
