// B3 + B4 fused for the NARROW blocks (cin <= 32, cout <= 64, dilation 1: the first SeperableConv block of every model, stride 1,
// and model 50's second, 32 -> 64 stride 2; posenet/models/mobilenet_v1.py:57-68), as warp-autonomous pipelines.
//
// In these blocks a 128-pixel tile carries so little work (128 x 32 x 9 depthwise MACs, a 128 x 64 x 32 GEMM) that the
// hand-offs of the CTA-wide pipeline in sepconv.cu (TMA -> depthwise warps -> tcgen05 -> epilogue warps, ~1.3k cycles of
// barrier latency per tile) cost more than the math.  Here every warp owns a column strip of 8 output pixels and walks
// down it on its own, with nothing shared between warps but the read-only weights:
//   * its lane 0 streams the strip's input rows (8 rows x 10 pixels x 32 channels per chunk, halo columns included, OOB
//     zero fill == the convolution's zero padding) into a private two-stage shared-memory ring with TMA;
//   * lanes 0-15 own the even pixels of the strip, lanes 16-31 the odd ones, one channel pair each (as the HALF mode of
//     sepconv.cu): the 3-row input window slides through registers as fp32 pairs, 36 packed FFMA2 per output row, same tap
//     order, bias, ReLU6 and bf16 rounding as dwconv.cu;
//   * two output rows (16 pixels) form one m16 tile: the depthwise result goes through a private 1.3 KB staging buffer
//     into mma.sync.m16n8k16 fragments (ldmatrix), the pointwise weights come from shared memory the same way, and the
//     fp32 accumulators get bias + ReLU6 and leave as 16-byte coalesced global stores (whole 128 B pixel rows).
// The GEMM is 1 % of a tcgen05 tile, so the legacy warp-level tensor path is the right size for it; no TMEM, no CTA barrier.
// Stride 2 (S = 2): a strip's 8 output pixels read 17 input columns and every output row two new input rows, so the chunks are
// 4 input rows x 17 pixels; of an output row's three input rows the last is carried over in registers (unpacked) as the next
// row's first and the other two pass through once.  (The CTA pipeline of sepconv.cu ran this block with half of every depthwise
// warp's lanes on zero-filled channels and one item per tile: 0.207 ms at 1281 x 721 x 32.)
// QTR (cin <= 16, model 50's first block): eight lanes cover a pixel's channel pairs, so a quarter-warp owns pixels q and q + 4
// of the strip instead of a half-warp owning every other pixel with half its lanes on zero-filled channels; the TMA box
// is 16 channels wide (32-byte pixels, so the four quarters still read 128 contiguous bytes).  Same taps in the same order.
#include <cuda.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "common.cuh"
#include "ptx.cuh"

namespace pn {

constexpr int SWP_WARPS = 16;
constexpr int SWP_THREADS = SWP_WARPS * 32;
constexpr int SWP_ROWS = 8;                               // input rows per TMA chunk
constexpr int SWP_COLS = 10;                              // 8 output pixels + 2 halo columns
constexpr int SWP_ROWS2 = 4, SWP_COLS2 = 17;              // stride 2: input rows per chunk, 2 * 8 + 1 input columns
constexpr int SWP_PIX = 64;                               // bytes per patch pixel (32 channels bf16)
constexpr int SWP_CHUNK = SWP_ROWS * SWP_COLS * SWP_PIX;  // 5120
constexpr int SWP_A_STRIDE = 80;                          // A staging: 16 pixel rows x (32 ch bf16 + 16 B pad), ldmatrix conflict-free
constexpr int SWP_O_STRIDE = 144;                         // output staging: 16 pixel rows x (64 ch bf16 + 16 B pad)
constexpr int SWP_W_STRIDE = 80;                          // pointwise weights [cout][32 + pad]
constexpr int SWP_WARP_SMEM = (2 * SWP_CHUNK + 16 * SWP_A_STRIDE + 16 * SWP_O_STRIDE + 16 + 127) / 128 * 128;   // 13952: TMA wants 128 B
constexpr int SWP_SHARED = 64 * SWP_W_STRIDE + 64 * 4;    // weights + bias
constexpr int SWP_SMEM = SWP_WARPS * SWP_WARP_SMEM + SWP_SHARED + 1024;

struct SwpGeom {
    int n, h, w, k, nc;            // h, w: OUTPUT rows / columns (= the input's for stride 1)
    int s;                         // stride (1 | 2)
    int full;                      // full-warp layout (cin 33..64, sepwarpf_kernel): strips of 4 pixels
    int strips, nq, rb;            // 8-pixel column strips per image row, row blocks per strip, output rows per block
    int ks, nt;                    // k16 slices (1 or 2), n8 tiles (cout / 8)
    int items;                     // n * strips * nq (< 2^31: 32-bit index arithmetic in the kernel)
};

__device__ __forceinline__ void ldmatrix_x4(uint32_t addr, uint32_t (&r)[4]) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void mma_bf16_16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t swp_lds_u32(uint32_t addr) {
    uint32_t r;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(r) : "r"(addr));
    return r;
}
__device__ __forceinline__ void swp_stg_v4_if(void *p, const uint4 &v, bool on) {          // one predicated STG.128, no branch
    if (on) asm volatile("st.global.v4.b32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void swp_sts_u32(uint32_t addr, uint32_t v) {
    asm volatile("st.shared.b32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}

// KS_T / NT_T: compile-time k16 slices and n8 tiles of the pointwise GEMM (0 = take them from the geometry at run time); the
// common widths get a fully unrolled tensor phase with immediate shared-memory offsets.
template <int KS_T, int NT_T, bool QTR = false, int S = 1>
__global__ void __launch_bounds__(SWP_THREADS, 1)
sepwarp_kernel(const __grid_constant__ CUtensorMap tmap_x, const float *__restrict__ dw_w, const float *__restrict__ dw_b,
               const __nv_bfloat16 *__restrict__ pw_w, const float *__restrict__ pw_b, __nv_bfloat16 *__restrict__ y, const SwpGeom g) {
    extern __shared__ uint8_t swp_raw[];
    const uint32_t base = (smem_u32(swp_raw) + 1023u) & ~1023u;
    uint8_t *gen = swp_raw + (base - smem_u32(swp_raw));
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t sW = base + SWP_WARPS * SWP_WARP_SMEM, sBias = sW + 64 * SWP_W_STRIDE;
    const uint32_t mine = base + (uint32_t)warp * SWP_WARP_SMEM;
    const uint32_t sRing = mine, sA = mine + 2 * SWP_CHUNK, sO = sA + 16 * SWP_A_STRIDE, bars = sO + 16 * SWP_O_STRIDE;

    // ---- CTA-wide, once: pointwise weights [cout][k] -> padded rows, bias; per warp: its two ring barriers
    for (int i = threadIdx.x; i < 64 * 4; i += SWP_THREADS) {            // (row n, 16-byte chunk c) = 8 input channels
        const int nrow = i >> 2, c = i & 3;
        uint4 v = make_uint4(0u, 0u, 0u, 0u);
        if (nrow < g.nc && c * 8 < g.k) v = *reinterpret_cast<const uint4 *>(pw_w + (size_t)nrow * g.k + c * 8);
        *reinterpret_cast<uint4 *>(gen + SWP_WARPS * SWP_WARP_SMEM + nrow * SWP_W_STRIDE + c * 16) = v;
    }
    if (threadIdx.x < 64) reinterpret_cast<float *>(gen + SWP_WARPS * SWP_WARP_SMEM + 64 * SWP_W_STRIDE)[threadIdx.x] =
        (int)threadIdx.x < g.nc ? pw_b[threadIdx.x] : 0.f;
    if (lane == 0) {
        mbar_init(bars, 1);
        mbar_init(bars + 8, 1);
        mbar_fence_init();
        if (warp == 0) tma_prefetch_desc(&tmap_x);
    }
    pdl_launch_dependents();
    __syncthreads();
    pdl_wait();                                                           // the weight staging above overlapped the stem's tail

    // ---- per lane: pixel parity, channel pair, the 9 x 2 depthwise weights + bias in registers for the whole kernel
    // NP pixels per lane, PSTEP strip pixels apart, NC window columns per row; window column of (pixel p, tap kx) = PSTEP p + kx
    // Stride 2 (S == 2; cin 17..32 -> the second block of model 50): a lane's four output pixels read input columns 4 p + kx
    // (+ 2 for the odd half), two new input rows per output row, chunks of 4 input rows x 17 columns.
    static_assert(S == 1 || (S == 2 && !QTR), "stride 2 uses the half-warp layout");
    constexpr int NP = QTR ? 2 : 4, PSTEP = QTR ? 4 : 2, NC = S == 2 ? 12 : QTR ? 6 : 9;
    constexpr bool COL4 = QTR || S == 2;                               // window column c sits at pixel (c / 3) * 4 + c % 3 (else at c)
    constexpr uint32_t PIXB = QTR ? 32u : (uint32_t)SWP_PIX;          // bytes per patch pixel (TMA box: 16 / 32 channels)
    constexpr int ROWS = S == 2 ? SWP_ROWS2 : SWP_ROWS, COLS = S == 2 ? SWP_COLS2 : SWP_COLS;
    constexpr uint32_t CHUNK_TX = ROWS * COLS * PIXB;                  // bytes a chunk's box delivers
    static_assert(SWP_ROWS2 * SWP_COLS2 * SWP_PIX <= SWP_CHUNK, "a stride-2 chunk fits the ring stage");
    const int hsel = QTR ? (lane >> 3) : (lane >> 4), cp = QTR ? (lane & 7) : (lane & 15);
    float2 wk[9], bias2;
    {
        const bool ok = 2 * cp < g.k;                                    // k is a multiple of 8: the pair is in or out as a whole
#pragma unroll
        for (int t = 0; t < 9; ++t) wk[t] = ok ? *reinterpret_cast<const float2 *>(dw_w + (size_t)t * g.k + 2 * cp) : make_float2(0.f, 0.f);
        bias2 = ok ? *reinterpret_cast<const float2 *>(dw_b + 2 * cp) : make_float2(0.f, 0.f);
    }
    auto unpack = [](uint32_t r) { return make_float2(__uint_as_float(r << 16), __uint_as_float(r & 0xffff0000u)); };
    const int ks_n = KS_T ? KS_T : g.ks, nt_n = NT_T ? NT_T : g.nt;
    const uint32_t lane_off = (uint32_t)(hsel * S) * PIXB + (uint32_t)cp * 4u;
    const uint32_t a_lane_addr = sA + (uint32_t)hsel * SWP_A_STRIDE + (uint32_t)cp * 4u;                 // + (half * 8 + 2 p) rows
    const uint32_t a_ld_addr = sA + (uint32_t)(lane & 15) * SWP_A_STRIDE + (uint32_t)(lane >> 4) * 16u;    // ldmatrix row / k-chunk
    const uint32_t w_ld_addr = sW + (uint32_t)(lane & 7) * SWP_W_STRIDE + (uint32_t)(lane >> 3) * 16u;     // + nt * 8 rows
    const int gq = lane >> 2, qq = lane & 3;                              // accumulator fragment: rows gq / gq + 8, columns 2 qq (+1)
    // the lane's pointwise bias pairs, one per n8 tile, in registers where the tile count is compile-time and the row-stationary
    // depthwise leaves room (stride 1): 8 shared-memory wavefronts less per 16 pixels (3.8 % of the kernel)
    constexpr bool BIAS_REG = NT_T > 0 && S == 1;
    float2 pbias[BIAS_REG ? NT_T : 1];
    if (BIAS_REG) {
#pragma unroll
        for (int nt = 0; nt < (BIAS_REG ? NT_T : 1); ++nt)
            asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(pbias[nt].x), "=f"(pbias[nt].y) : "r"(sBias + (uint32_t)(nt * 8 + 2 * qq) * 4u));
    }

    uint32_t phase_bits = 0;                                              // bit s = parity of ring stage s
    uint32_t chunk_ctr = 0;                                               // chunks this warp has consumed so far (stage = ctr & 1)
    const int total_warps = (int)gridDim.x * SWP_WARPS, first_item = (int)blockIdx.x * SWP_WARPS + warp;

    // item -> (image, row block, strip); consecutive warps take neighbouring strips (they share halo columns in L2)
    struct Item { int x0, y0, img, rows_out, nchunks; };
    auto decode = [&](int it) {
        Item t;
        const int xs = it % g.strips, rest = it / g.strips;
        t.x0 = xs * 8;
        t.y0 = (rest % g.nq) * g.rb;
        t.img = rest / g.nq;
        t.rows_out = min(g.rb, g.h - t.y0);
        t.nchunks = t.rows_out > 0 ? (S * t.rows_out + 3 - S + ROWS - 1) / ROWS : 0;     // input rows: S (rows_out - 1) + 3
        return t;
    };
    // Lane 0 runs a producer cursor two chunks ahead of the consumer, across item boundaries, so the ring does not drain
    // between items.
    int p_item = first_item, p_ci = 0;
    uint32_t p_chunks = 0;                                                // chunks issued so far (stage = count & 1)
    Item pit = p_item < g.items ? decode(p_item) : Item{0, 0, 0, 0, 0};
    auto issue_next = [&]() {                                             // lane 0: the next chunk in (item, chunk) order, if any
        while (p_item < g.items && p_ci >= pit.nchunks) {
            p_item += total_warps;
            p_ci = 0;
            if (p_item < g.items) pit = decode(p_item);
        }
        if (p_item >= g.items) return;
        const uint32_t s_ = p_chunks & 1u;
        mbar_expect_tx(bars + 8u * s_, CHUNK_TX);
        tma_load_4d(sRing + s_ * SWP_CHUNK, &tmap_x, bars + 8u * s_, 0, S * pit.x0 - 1, S * pit.y0 - 1 + p_ci * ROWS, pit.img);
        ++p_chunks;
        ++p_ci;
    };
    if (lane == 0) {
        issue_next();
        issue_next();
    }

    for (int item = first_item; item < g.items; item += total_warps) {
        const Item it = decode(item);
        const int x0 = it.x0, y0 = it.y0, img = it.img, rows_out = it.rows_out;
        if (rows_out <= 0) continue;
        const int rows_in = S * (rows_out - 1) + 3;
        const int ncol_ok = g.w - x0;                                     // strip pixels px < ncol_ok exist
        // output addressing for the 16-byte stores of the tensor phase: lane -> (pixel lane >> 3 (+4), 8 channels lane & 7); one
        // 64-bit pointer per lane, advanced by two output rows per phase
        const size_t pix_bytes = (size_t)g.nc * 2, row_bytes = (size_t)g.w * pix_bytes;
        char *o_pair = reinterpret_cast<char *>(y) + ((((size_t)img * g.h + y0) * g.w + (x0 + (lane >> 3))) * g.nc + (lane & 7) * 8) * 2;
        const bool ok_lo = (lane & 7) < nt_n && (lane >> 3) < ncol_ok, ok_hi = (lane & 7) < nt_n && (lane >> 3) + 4 < ncol_ok;
        const uint32_t so_lane = sO + (uint32_t)(lane >> 3) * SWP_O_STRIDE + (uint32_t)(lane & 7) * 16u;
        uint32_t stage_addr = 0;
        // input row r of the item: wait for its chunk when it is the chunk's first row; returns the lane's address of the row
        auto enter_row = [&](const int r) {
            const uint32_t ci = (uint32_t)r / (uint32_t)ROWS, rr = (uint32_t)r % (uint32_t)ROWS;    // (ROWS is a power of two)
            if (rr == 0) {
                const uint32_t s_ = (chunk_ctr + ci) & 1u;
                mbar_wait(bars + 8u * s_, (phase_bits >> s_) & 1u);
                phase_bits ^= 1u << s_;
                stage_addr = sRing + s_ * SWP_CHUNK + lane_off;
            }
            return stage_addr + rr * (uint32_t)(COLS * PIXB);
        };
        // ... and once the chunk's last row is in registers (its FMAs issued by every lane) the stage is refilled
        auto leave_row = [&](const int r) {
            if (((uint32_t)r & (uint32_t)(ROWS - 1)) == (uint32_t)(ROWS - 1) || r == rows_in - 1) {
                __syncwarp();
                if (lane == 0) issue_next();                              // (of this item or the next)
            }
        };
        auto load_row = [&](const uint32_t rp, float2 (&row)[NC]) {
#pragma unroll
            for (int c = 0; c < NC; ++c) row[c] = unpack(swp_lds_u32(rp + (uint32_t)(COL4 ? (c / 3) * 4 + c % 3 : c) * PIXB));
        };
        auto fma_row = [&](const float2 (&row)[NC], const int ky, float2 (&acc)[NP]) {   // taps (ky, 0..2) of every pixel, kx ascending
#pragma unroll
            for (int c = 0; c < NC; ++c)
#pragma unroll
                for (int p = 0; p < NP; ++p)
#pragma unroll
                    for (int kx = 0; kx < 3; ++kx)
                        if ((COL4 ? 3 * p + kx : 2 * p + kx) == c) acc[p] = ffma2(row[c], wk[ky * 3 + kx], acc[p]);
        };
        // depthwise row t of the item -> A staging; after two rows (or the last single one): 16 pixels x cin -> pointwise GEMM on
        // mma.sync -> output staging -> 16-byte coalesced stores
        auto finish_row = [&](const int t, const float2 (&acc)[NP]) {
            const uint32_t arow = a_lane_addr + (uint32_t)((t & 1) * 8) * SWP_A_STRIDE;
#pragma unroll
            for (int p = 0; p < NP; ++p) swp_sts_u32(arow + (uint32_t)(PSTEP * p) * SWP_A_STRIDE, relu6_bf16x2(acc[p]));
            if (!((t & 1) || t == rows_out - 1)) return;
            __syncwarp();
            uint32_t a0[4], a1[4] = {0u, 0u, 0u, 0u};
            ldmatrix_x4(a_ld_addr, a0);
            if (ks_n > 1) ldmatrix_x4(a_ld_addr + 32u, a1);
            auto tile_n = [&](const int nt) {
                uint32_t b[4];
                ldmatrix_x4(w_ld_addr + (uint32_t)(nt * 8) * SWP_W_STRIDE, b);
                float d[4] = {0.f, 0.f, 0.f, 0.f};
                mma_bf16_16816(d, a0, b[0], b[1]);
                if (ks_n > 1) mma_bf16_16816(d, a1, b[2], b[3]);
                float2 bv;
                if (BIAS_REG) bv = pbias[BIAS_REG ? nt : 0];
                else asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(bv.x), "=f"(bv.y) : "r"(sBias + (uint32_t)(nt * 8 + 2 * qq) * 4u));
                const uint32_t o = sO + (uint32_t)gq * SWP_O_STRIDE + (uint32_t)(nt * 16 + qq * 4);
                swp_sts_u32(o, relu6_bf16x2(fadd2(make_float2(d[0], d[1]), bv)));
                swp_sts_u32(o + 8u * SWP_O_STRIDE, relu6_bf16x2(fadd2(make_float2(d[2], d[3]), bv)));
            };
            if (NT_T) {
#pragma unroll
                for (int nt = 0; nt < (NT_T ? NT_T : 1); ++nt) tile_n(nt);
            } else {
#pragma unroll 2
                for (int nt = 0; nt < nt_n; ++nt) tile_n(nt);
            }
            __syncwarp();
            // 8 lanes cover one pixel's channels, 4 pixels per instruction (staging row = output-row parity * 8 + pixel); the
            // second row exists when the pair is complete
            const bool two = (t & 1) != 0;
            char *o1 = o_pair + 4 * pix_bytes, *o2 = o_pair + row_bytes, *o3 = o2 + 4 * pix_bytes;
            swp_stg_v4_if(o_pair, ld_shared_v4(so_lane), ok_lo);
            swp_stg_v4_if(o1, ld_shared_v4(so_lane + 4u * SWP_O_STRIDE), ok_hi);
            swp_stg_v4_if(o2, ld_shared_v4(so_lane + 8u * SWP_O_STRIDE), ok_lo && two);
            swp_stg_v4_if(o3, ld_shared_v4(so_lane + 12u * SWP_O_STRIDE), ok_hi && two);
            o_pair += 2 * row_bytes;
            __syncwarp();                                                 // staging buffers are rewritten by the next rows
        };
        if constexpr (S == 1) {
            // Row-stationary: an input row is unpacked once and feeds the three output rows it belongs to -- as the first window row
            // of output r (whose accumulators start from the bias here), the second of r - 1, the third of r - 2, which is then
            // complete.  Three sets of accumulators instead of a three-row window (24 instead of 54 registers; the ones saved hold
            // the pointwise bias), and every accumulator still sees bias, (ky 0: kx 0 1 2), (ky 1: ..), (ky 2: ..) in that order.
            // Rows 0 and 1 also add into sets that stand for output rows -1 / -2: those are re-initialised before they are used.
            float2 accs[3][NP];
#pragma unroll
            for (int j = 0; j < 3; ++j)
#pragma unroll
                for (int p = 0; p < NP; ++p) accs[j][p] = bias2;
#pragma unroll 1
            for (int r0 = 0; r0 < rows_in; r0 += 3) {
#pragma unroll
                for (int j = 0; j < 3; ++j) {
                    const int r = r0 + j;
                    if (r >= rows_in) break;
                    float2 row[NC];
                    load_row(enter_row(r), row);
#pragma unroll
                    for (int p = 0; p < NP; ++p) accs[j][p] = bias2;
                    fma_row(row, 0, accs[j]);
                    fma_row(row, 1, accs[(j + 2) % 3]);
                    fma_row(row, 2, accs[(j + 1) % 3]);
                    if (r < 2) continue;                                  // (rows_in >= 3: no refill point among rows 0, 1)
                    finish_row(r - 2, accs[(j + 1) % 3]);
                    leave_row(r);
                }
            }
        } else {
            // output row t reads input rows 2t, 2t + 1, 2t + 2: the last one is carried over (unpacked) as the next row's first,
            // the other two pass through registers once.  Same tap order as every other depthwise kernel (ky outer, kx inner).
            float2 carry[NC], tmp[NC];
            load_row(enter_row(0), carry);
#pragma unroll 1
            for (int t = 0; t < rows_out; ++t) {
                float2 acc[NP];
#pragma unroll
                for (int p = 0; p < NP; ++p) acc[p] = bias2;
                fma_row(carry, 0, acc);
                load_row(enter_row(2 * t + 1), tmp);
                fma_row(tmp, 1, acc);
                leave_row(2 * t + 1);
                load_row(enter_row(2 * t + 2), carry);
                fma_row(carry, 2, acc);
                finish_row(t, acc);
                leave_row(2 * t + 2);
            }
        }
        chunk_ctr += (uint32_t)it.nchunks;
    }
}

// ---- full-warp layout: cin 33..64 -------------------------------------------------------------------------------------
// The same warp-autonomous pipeline for blocks whose channel pairs fill a whole warp (lane = channel pair, like dwwarp.cu):
// a strip is 4 output pixels wide, four output rows form the m16 tile, the GEMM has KS k16 slices and NT n8 tiles (all
// compile-time: one instantiation per block shape that measured faster than the CTA pipeline of sepconv.cu -- 48 -> 96
// stride 2, the second block of model 75, which ran there with a quarter of its depthwise lanes on zero-filled channels:
// 0.293 -> 0.272 ms at 129 x 129 x 512).  Chunks are 4 input rows; the TMA box is as wide as cin rounded up to 16
// channels, so a 48-channel pixel is 96 bytes.  Same taps in the same order as every other depthwise kernel.
template <int KS, int NT, int S> struct SwfCfg {
    static constexpr int PIXB = KS * 32;                       // bytes per patch pixel
    static constexpr int ROWS = 4, COLS = S == 2 ? 9 : 6;      // input rows per chunk; 4 output pixels -> 2 * 4 + 1 | 4 + 2 input columns
    static constexpr int CHUNK = ROWS * COLS * PIXB;           // (a multiple of 128: KS * 32 * 4 = KS * 128)
    static constexpr int A_STRIDE = PIXB + 16, O_STRIDE = NT * 16 + 16, W_STRIDE = PIXB + 16;   // odd numbers of 16-byte chunks: conflict-free
    static constexpr int WARP_SMEM = (2 * CHUNK + 16 * A_STRIDE + 16 * O_STRIDE + 16 + 127) / 128 * 128;
    static constexpr int SHARED = NT * 8 * W_STRIDE + NT * 8 * 4;
    static constexpr int SMEM = SWP_WARPS * WARP_SMEM + SHARED + 1024;
    static_assert(SMEM <= 227 * 1024, "shared memory");
};

template <int KS, int NT, int S>
__global__ void __launch_bounds__(SWP_THREADS, 1)
sepwarpf_kernel(const __grid_constant__ CUtensorMap tmap_x, const float *__restrict__ dw_w, const float *__restrict__ dw_b,
                const __nv_bfloat16 *__restrict__ pw_w, const float *__restrict__ pw_b, __nv_bfloat16 *__restrict__ y, const SwpGeom g) {
    using Cfg = SwfCfg<KS, NT, S>;
    constexpr uint32_t PIXB = Cfg::PIXB, CHUNK = Cfg::CHUNK, A_STRIDE = Cfg::A_STRIDE, O_STRIDE = Cfg::O_STRIDE, W_STRIDE = Cfg::W_STRIDE;
    constexpr int ROWS = Cfg::ROWS, COLS = Cfg::COLS, NC = COLS;
    extern __shared__ uint8_t swp_raw[];
    const uint32_t base = (smem_u32(swp_raw) + 1023u) & ~1023u;
    uint8_t *gen = swp_raw + (base - smem_u32(swp_raw));
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t sW = base + SWP_WARPS * Cfg::WARP_SMEM, sBias = sW + NT * 8 * W_STRIDE;
    const uint32_t mine = base + (uint32_t)warp * Cfg::WARP_SMEM;
    const uint32_t sRing = mine, sA = mine + 2 * CHUNK, sO = sA + 16 * A_STRIDE, bars = sO + 16 * O_STRIDE;

    // ---- CTA-wide, once: pointwise weights [cout][k] -> padded rows (channels beyond cin zero), bias; per warp: its ring barriers
    for (int i = threadIdx.x; i < NT * 8 * KS * 2; i += SWP_THREADS) {   // (row n, 16-byte chunk c) = 8 input channels
        const int nrow = i / (KS * 2), c = i - nrow * (KS * 2);
        uint4 v = make_uint4(0u, 0u, 0u, 0u);
        if (nrow < g.nc && c * 8 < g.k) v = *reinterpret_cast<const uint4 *>(pw_w + (size_t)nrow * g.k + c * 8);
        *reinterpret_cast<uint4 *>(gen + SWP_WARPS * Cfg::WARP_SMEM + nrow * W_STRIDE + c * 16) = v;
    }
    if (threadIdx.x < NT * 8) reinterpret_cast<float *>(gen + SWP_WARPS * Cfg::WARP_SMEM + NT * 8 * W_STRIDE)[threadIdx.x] =
        (int)threadIdx.x < g.nc ? pw_b[threadIdx.x] : 0.f;
    if (lane == 0) {
        mbar_init(bars, 1);
        mbar_init(bars + 8, 1);
        mbar_fence_init();
        if (warp == 0) tma_prefetch_desc(&tmap_x);
    }
    pdl_launch_dependents();
    __syncthreads();
    pdl_wait();

    // ---- per lane: its channel pair's 9 x 2 depthwise weights + bias; lanes beyond cin / 2 compute on channel pair 0 and store nothing
    const bool lane_on = 2 * lane < g.k;
    const int cp = lane_on ? lane : 0;
    float2 wk[9], bias2;
#pragma unroll
    for (int t = 0; t < 9; ++t) wk[t] = *reinterpret_cast<const float2 *>(dw_w + (size_t)t * g.k + 2 * cp);
    bias2 = *reinterpret_cast<const float2 *>(dw_b + 2 * cp);
    auto unpack = [](uint32_t r) { return make_float2(__uint_as_float(r << 16), __uint_as_float(r & 0xffff0000u)); };
    const uint32_t lane_off = (uint32_t)cp * 4u;
    const uint32_t a_lane_addr = sA + (uint32_t)cp * 4u;                                                  // + (4 (t & 3) + p) rows
    const uint32_t a_ld_addr = sA + (uint32_t)(lane & 15) * A_STRIDE + (uint32_t)(lane >> 4) * 16u;         // ldmatrix row / k-chunk
    const uint32_t w_ld_addr = sW + (uint32_t)(lane & 7) * W_STRIDE + (uint32_t)(lane >> 3) * 16u;          // + nt * 8 rows
    const int gq = lane >> 2, qq = lane & 3;                              // accumulator fragment: rows gq / gq + 8, columns 2 qq (+1)

    uint32_t phase_bits = 0, chunk_ctr = 0;
    const int total_warps = (int)gridDim.x * SWP_WARPS, first_item = (int)blockIdx.x * SWP_WARPS + warp;
    struct Item { int x0, y0, img, rows_out, nchunks; };
    auto decode = [&](int it) {
        Item t;
        const int xs = it % g.strips, rest = it / g.strips;
        t.x0 = xs * 4;
        t.y0 = (rest % g.nq) * g.rb;
        t.img = rest / g.nq;
        t.rows_out = min(g.rb, g.h - t.y0);
        t.nchunks = t.rows_out > 0 ? (S * t.rows_out + 3 - S + ROWS - 1) / ROWS : 0;     // input rows: S (rows_out - 1) + 3
        return t;
    };
    int p_item = first_item, p_ci = 0;
    uint32_t p_chunks = 0;
    Item pit = p_item < g.items ? decode(p_item) : Item{0, 0, 0, 0, 0};
    auto issue_next = [&]() {                                             // lane 0: the next chunk in (item, chunk) order, if any
        while (p_item < g.items && p_ci >= pit.nchunks) {
            p_item += total_warps;
            p_ci = 0;
            if (p_item < g.items) pit = decode(p_item);
        }
        if (p_item >= g.items) return;
        const uint32_t s_ = p_chunks & 1u;
        mbar_expect_tx(bars + 8u * s_, CHUNK);
        tma_load_4d(sRing + s_ * CHUNK, &tmap_x, bars + 8u * s_, 0, S * pit.x0 - 1, S * pit.y0 - 1 + p_ci * ROWS, pit.img);
        ++p_chunks;
        ++p_ci;
    };
    if (lane == 0) {
        issue_next();
        issue_next();
    }

    for (int item = first_item; item < g.items; item += total_warps) {
        const Item it = decode(item);
        const int x0 = it.x0, y0 = it.y0, img = it.img, rows_out = it.rows_out;
        if (rows_out <= 0) continue;
        const int rows_in = S * (rows_out - 1) + 3;
        const int ncol_ok = g.w - x0;                                     // strip pixels px < ncol_ok exist
        const size_t pix_bytes = (size_t)g.nc * 2, row_bytes = (size_t)g.w * pix_bytes;
        // output stores of the tensor phase: 16-byte chunk q = i * 32 + lane of the 16 x NT chunks of an m16 tile belongs to staging
        // row q / NT (= 4 * tile row + pixel) and channels 8 (q % NT) ..; the pointer advances by four output rows per phase
        char *o_tile = reinterpret_cast<char *>(y) + (((size_t)img * g.h + y0) * g.w + x0) * pix_bytes;
        uint32_t stage_addr = 0;
        auto enter_row = [&](const int r) {
            const uint32_t ci = (uint32_t)r / (uint32_t)ROWS, rr = (uint32_t)r % (uint32_t)ROWS;    // (ROWS is a power of two)
            if (rr == 0) {
                const uint32_t s_ = (chunk_ctr + ci) & 1u;
                mbar_wait(bars + 8u * s_, (phase_bits >> s_) & 1u);
                phase_bits ^= 1u << s_;
                stage_addr = sRing + s_ * CHUNK + lane_off;
            }
            return stage_addr + rr * (uint32_t)(COLS * PIXB);
        };
        auto leave_row = [&](const int r) {
            if (((uint32_t)r & (uint32_t)(ROWS - 1)) == (uint32_t)(ROWS - 1) || r == rows_in - 1) {
                __syncwarp();
                if (lane == 0) issue_next();
            }
        };
        auto load_row = [&](const uint32_t rp, float2 (&row)[NC]) {
#pragma unroll
            for (int c = 0; c < NC; ++c) row[c] = unpack(swp_lds_u32(rp + (uint32_t)c * PIXB));
        };
        auto fma_row = [&](const float2 (&row)[NC], const int ky, float2 (&acc)[4]) {   // taps (ky, 0..2) of every pixel, kx ascending
#pragma unroll
            for (int c = 0; c < NC; ++c)
#pragma unroll
                for (int p = 0; p < 4; ++p)
#pragma unroll
                    for (int kx = 0; kx < 3; ++kx)
                        if (S * p + kx == c) acc[p] = ffma2(row[c], wk[ky * 3 + kx], acc[p]);
        };
        auto finish_row = [&](const int t, const float2 (&acc)[4]) {
            const uint32_t arow = a_lane_addr + (uint32_t)((t & 3) * 4) * A_STRIDE;
            if (lane_on) {
#pragma unroll
                for (int p = 0; p < 4; ++p) swp_sts_u32(arow + (uint32_t)p * A_STRIDE, relu6_bf16x2(acc[p]));
            }
            if (!((t & 3) == 3 || t == rows_out - 1)) return;
            // ---- four output rows (or the last 1-3) are staged: 16 pixels x cin -> pointwise GEMM on mma.sync
            __syncwarp();
            uint32_t a[KS][4];
#pragma unroll
            for (int ks = 0; ks < KS; ++ks) ldmatrix_x4(a_ld_addr + (uint32_t)ks * 32u, a[ks]);
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                uint32_t b[(KS + 1) / 2][4];
#pragma unroll
                for (int h2 = 0; h2 < (KS + 1) / 2; ++h2) ldmatrix_x4(w_ld_addr + (uint32_t)(nt * 8) * W_STRIDE + (uint32_t)h2 * 64u, b[h2]);
                float d[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                for (int ks = 0; ks < KS; ++ks) mma_bf16_16816(d, a[ks], b[ks >> 1][(ks & 1) * 2], b[ks >> 1][(ks & 1) * 2 + 1]);
                float2 bv;
                asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(bv.x), "=f"(bv.y) : "r"(sBias + (uint32_t)(nt * 8 + 2 * qq) * 4u));
                const uint32_t o = sO + (uint32_t)gq * O_STRIDE + (uint32_t)(nt * 16 + qq * 4);
                swp_sts_u32(o, relu6_bf16x2(fadd2(make_float2(d[0], d[1]), bv)));
                swp_sts_u32(o + 8u * O_STRIDE, relu6_bf16x2(fadd2(make_float2(d[2], d[3]), bv)));
            }
            __syncwarp();
            const int nrows = (t & 3) + 1;                                // tile rows that exist
#pragma unroll
            for (int i = 0; i < (16 * NT + 31) / 32; ++i) {
                const int q = i * 32 + lane, px = q / NT, ch = q - px * NT, trow = px >> 2, tcol = px & 3;
                const bool ok = q < 16 * NT && trow < nrows && tcol < ncol_ok;
                swp_stg_v4_if(o_tile + (size_t)trow * row_bytes + (size_t)tcol * pix_bytes + (size_t)ch * 16,
                              ld_shared_v4(sO + (uint32_t)px * O_STRIDE + (uint32_t)ch * 16u), ok);
            }
            o_tile += 4 * row_bytes;
            __syncwarp();                                                 // staging buffers are rewritten by the next rows
        };
        if constexpr (S == 1) {
            float2 ring[3][NC];                                           // input rows r-2, r-1, r live in slots (j+1)%3, (j+2)%3, j
#pragma unroll 1
            for (int r0 = 0; r0 < rows_in; r0 += 3) {
#pragma unroll
                for (int j = 0; j < 3; ++j) {
                    const int r = r0 + j;
                    if (r >= rows_in) break;
                    load_row(enter_row(r), ring[j]);
                    if (r < 2) continue;
                    float2 acc[4] = {bias2, bias2, bias2, bias2};
#pragma unroll
                    for (int ky = 0; ky < 3; ++ky) fma_row(ring[(j + 1 + ky) % 3], ky, acc);
                    finish_row(r - 2, acc);
                    leave_row(r);
                }
            }
        } else {
            float2 carry[NC], tmp[NC];                                    // (see sepwarp_kernel: the shared input row is carried over)
            load_row(enter_row(0), carry);
#pragma unroll 1
            for (int t = 0; t < rows_out; ++t) {
                float2 acc[4] = {bias2, bias2, bias2, bias2};
                fma_row(carry, 0, acc);
                load_row(enter_row(2 * t + 1), tmp);
                fma_row(tmp, 1, acc);
                leave_row(2 * t + 1);
                load_row(enter_row(2 * t + 2), carry);
                fma_row(carry, 2, acc);
                finish_row(t, acc);
                leave_row(2 * t + 2);
            }
        }
        chunk_ctr += (uint32_t)it.nchunks;
    }
}

// ---- host side ---------------------------------------------------------------------------------------------
// block shapes with an instantiation of the full-warp kernel (measured against the CTA pipeline on the blocks of models 75 / 50)
static bool sepwarp_full_shape(int k, int nc, int stride) {
    // (64 -> 64 stride 1, the third block of model 50, was measured too -- sepwarpf_kernel<4, 8, 1>: 0.164 vs 0.160 ms on the CTA
    // pipeline at 181 x 321 x 32 -- and stays there)
    return k == 48 && nc == 96 && stride == 2;
}

bool sepwarp_supported(int k, int nc, int stride, int dil) {
    if (dil == 1 && sepwarp_full_shape(k, nc, stride)) return true;
    if (!(dil == 1 && k >= 8 && k <= 32 && k % 8 == 0 && nc >= 8 && nc <= 64 && nc % 8 == 0)) return false;
    // stride 2: cin 17..32 (the half-warp layout; narrower blocks would idle half its lanes)
    return stride == 1 || (stride == 2 && k > 16);
}

// strips / row blocks / item count: pure host arithmetic (no CUDA calls beyond the cached SM count); h, wd: the INPUT map
int sepwarp_geometry(SepWarpOp *op, int n, int h, int wd, int k, int nc, int stride) {
    PN_CHECK_ARG(n > 0 && h > 0 && wd > 0 && sepwarp_supported(k, nc, stride, 1), "pn_sepconv_block: bad narrow-block shape");
    memset(op, 0, sizeof(*op));
    SwpGeom g;
    memset(&g, 0, sizeof(g));
    g.n = n; g.k = k; g.nc = nc; g.s = stride;
    g.h = (h - 1) / stride + 1;                                            // 3x3, pad 1: floor((h + 2 - 3) / s) + 1
    g.w = (wd - 1) / stride + 1;
    g.full = sepwarp_full_shape(k, nc, stride) ? 1 : 0;
    g.strips = ceil_div(g.w, g.full ? 4 : 8);
    g.ks = ceil_div(k, 16);
    g.nt = nc / 8;
    // Row blocks.  Items go to the warps of a full grid round-robin (item i -> warp i mod W, strips fastest), a warp walks its
    // items one after the other, and an item costs its input rows (measured: the time of a launch follows the LARGEST per-warp sum
    // of input rows within 2 % across row-block counts; the per-item overhead is nil).  With only a handful of items per warp the
    // quantisation of that sum is worth 5-20 %, so every row-block count (blocks of at least 8 output rows) is simulated and the
    // best one taken: 64 x 257 x 257: 7 -> 10 blocks, 512 x 129 x 129: 2 -> 4, 32 x 361 x 641 stride 2: 11 -> 7.
    const int warps = num_sms() * SWP_WARPS;
    const int max_nq = ceil_div(g.h, 8);
    long long nq = 1;
    std::vector<long long> load((size_t)warps);
    long long best = -1;
    for (int cand = 1; cand <= max_nq; ++cand) {
        const int rb = ceil_div(g.h, cand);
        if (ceil_div(g.h, rb) != cand) continue;                           // (the same blocks as a smaller count)
        const long long items_c = (long long)n * g.strips * cand;
        if (items_c > (1ll << 22)) break;                                  // (plan-time work bound; never reached by the reference's sizes)
        std::fill(load.begin(), load.end(), 0ll);
        int wi = 0, xs = 0, q = 0;
        for (long long it = 0; it < items_c; ++it) {
            load[(size_t)wi] += (long long)(rb < g.h - q * rb ? rb : g.h - q * rb) * stride + (3 - stride);
            if (++wi == warps) wi = 0;
            if (++xs == g.strips) { xs = 0; if (++q == cand) q = 0; }
        }
        const long long worst = *std::max_element(load.begin(), load.end());
        if (best < 0 || worst < best) { best = worst; nq = cand; }
    }
    g.rb = ceil_div(g.h, (int)nq);
    g.nq = ceil_div(g.h, g.rb);
    const long long items = (long long)n * g.strips * g.nq;
    PN_CHECK_ARG(items + (long long)num_sms() * SWP_WARPS < (1ll << 31), "pn_sepconv_block: problem too large for one launch");
    g.items = (int)items;
    static_assert(sizeof(SwpGeom) <= sizeof(op->geom), "SepWarpOp::geom too small");
    memcpy(op->geom, &g, sizeof(g));
    return PN_OK;
}

int sepwarp_prepare(SepWarpOp *op, const void *x, int n, int h, int wd, int k, int nc, int stride) {
    int rc = sepwarp_geometry(op, n, h, wd, k, nc, stride);
    if (rc != PN_OK) return rc;
    const uint64_t dims[4] = {(uint64_t)k, (uint64_t)wd, (uint64_t)h, (uint64_t)n};
    const uint64_t strides[3] = {(uint64_t)k * 2, (uint64_t)wd * k * 2, (uint64_t)h * wd * k * 2};
    // (k <= 16, stride 1: the QTR kernel's 32-byte pixels; stride 2: chunks of 4 input rows x 17 columns)
    const uint32_t box[4] = {(k <= 16 && stride == 1) ? 16u : 32u, (uint32_t)(stride == 2 ? SWP_COLS2 : SWP_COLS),
                             (uint32_t)(stride == 2 ? SWP_ROWS2 : SWP_ROWS), 1u};
    if (sepwarp_full_shape(k, nc, stride)) {                             // full-warp layout: cin rounded up to 16 channels, 4-pixel strips, 4-row chunks
        const uint32_t fbox[4] = {(uint32_t)ceil_div(k, 16) * 16u, (uint32_t)(stride == 2 ? 9 : 6), 4u, 1u};
        return encode_tmap(op->tmap_x, x, 2, 4, dims, strides, fbox, 0);
    }
    return encode_tmap(op->tmap_x, x, 2, 4, dims, strides, box, 0);
}

int sepwarp_launch(const SepWarpOp *op, const float *dw_w, const float *dw_b, const void *pw_w, const float *pw_b, void *y,
                   cudaStream_t st) {
    PN_CHECK_ARG(op && dw_w && dw_b && pw_w && pw_b && y, "pn_sepconv_block: null pointer");
    PN_CHECK_ARG(((uintptr_t)y & 15) == 0 && ((uintptr_t)pw_w & 15) == 0 && ((uintptr_t)dw_w & 7) == 0 && ((uintptr_t)dw_b & 7) == 0,
                 "pn_sepconv_block: misaligned pointer");
    SwpGeom g;
    memcpy(&g, op->geom, sizeof(g));
    const long long ctas = ((long long)g.items + SWP_WARPS - 1) / SWP_WARPS;
    const int grid = (int)(ctas < num_sms() ? ctas : num_sms());
    const int dev = current_device();
    auto launch = [&](auto kern, DeviceOnce &once) -> int {
        if (!once.get(dev)) {
            PN_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SWP_SMEM));
            once.set(dev, 1);
        }
        PN_CHECK_CUDA(launch_pdl(kern, dim3(grid), dim3(SWP_THREADS), SWP_SMEM, st, *reinterpret_cast<const CUtensorMap *>(op->tmap_x), dw_w, dw_b,
                                 (const __nv_bfloat16 *)pw_w, pw_b, (__nv_bfloat16 *)y, g));
        return PN_OK;
    };
    if (g.full) {
        auto launch_f = [&](auto kern, int smem, DeviceOnce &once) -> int {
            if (!once.get(dev)) {
                PN_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
                once.set(dev, 1);
            }
            PN_CHECK_CUDA(launch_pdl(kern, dim3(grid), dim3(SWP_THREADS), (size_t)smem, st, *reinterpret_cast<const CUtensorMap *>(op->tmap_x), dw_w,
                                     dw_b, (const __nv_bfloat16 *)pw_w, pw_b, (__nv_bfloat16 *)y, g));
            return PN_OK;
        };
        static DeviceOnce f3122;
        if (g.k == 48 && g.nc == 96 && g.s == 2) return launch_f(sepwarpf_kernel<3, 12, 2>, SwfCfg<3, 12, 2>::SMEM, f3122);   // model 75, block 2
        set_error("pn_sepconv_block: no full-warp instantiation for %d -> %d stride %d", g.k, g.nc, g.s);
        return PN_ERR_UNSUPPORTED;
    }
    static DeviceOnce c28, c26, c14, c00, c00q, s28, s00;
    if (g.s == 2) {
        if (g.ks == 2 && g.nt == 8) return launch(sepwarp_kernel<2, 8, false, 2>, s28);   // 32 -> 64 stride 2 (model 50)
        return launch(sepwarp_kernel<0, 0, false, 2>, s00);
    }
    if (g.ks == 2 && g.nt == 8) return launch(sepwarp_kernel<2, 8>, c28);      // 32 -> 64 (model 100 / 101)
    if (g.ks == 2 && g.nt == 6) return launch(sepwarp_kernel<2, 6>, c26);      // 24 -> 48 (model 75)
    if (g.ks == 1 && g.nt == 4) return launch(sepwarp_kernel<1, 4, true>, c14);      // 16 -> 32 (model 50)
    if (g.k <= 16) return launch(sepwarp_kernel<0, 0, true>, c00q);
    return launch(sepwarp_kernel<0, 0>, c00);
}

void sepwarp_describe(const SepWarpOp *op, char *out, size_t cap) {
    SwpGeom g;
    memcpy(&g, op->geom, sizeof(g));
    snprintf(out, cap, "warp-autonomous%s%s strips %d x %d row blocks of %d rows, k16 slices %d, n8 tiles %d, items %d, smem %d",
             g.full ? " full-warp" : "", g.s == 2 ? " stride 2" : "", g.strips, g.nq, g.rb, g.ks, g.nt, g.items, SWP_SMEM);
}

}  // namespace pn
