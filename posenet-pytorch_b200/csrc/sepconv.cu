// B3 + B4 fused -- one whole SeperableConv block (posenet/models/mobilenet_v1.py:57-68 of the reference):
//     y = relu6( pointwise1x1( relu6( depthwise3x3(x; stride, dilation) + b_dw ) ) + b_pw )
// as ONE kernel: the depthwise result never travels to HBM.  It is produced by CUDA-core warps straight
// into the 128B-swizzled shared-memory A tile that the tcgen05 tensor-core GEMM of the pointwise conv reads.
//
// Work item: an output tile of TH x TW (<= 128) pixels of one image x N_TILE (<= 256) output channels.
// Per 64-channel k-block of the tile (persistent CTA, 1 per SM, warp-specialised):
//   warp 0      TMA producer   input patch incl. halo as ONE cp.async.bulk.tensor.4d box per sub-tile (OOB zero fill
//                              == the convolution's zero padding), the k-block's depthwise weights + bias ([9,K] /
//                              [K] fp32 through 2-D maps, ragged K zero-filled), and the pointwise weight tile
//                              [N_TILE x 64] (128B swizzle) -- three mbarrier rings (patch / W / A).
//   warps 6-15  depthwise      a lane owns one channel pair (4 B of every pixel), a warp a column strip of 4 output pixels
//                              (segments are handed out dynamically from a shared-memory counter, so the warps of the four
//                              schedulers stay busy and run ahead into the next k-block while others finish the current one)
//                              that it walks down row by row with the 3x3 window's input rows held in registers, so
//                              each patch element is read from shared memory once and the 9x2 weights stay in
//                              registers (the kernel is shared-memory-bandwidth bound otherwise).  fp32 math with packed
//                              fma.rn.f32x2 in the same tap order as the stand-alone kernel (dwconv.cu), + bias, ReLU6,
//                              -> bf16 -> st.shared into row r = ty*TW+tx of the A stage (16-byte chunk index XOR
//                              (r & 7) = SWIZZLE_128B K-major), fence.proxy.async, mbarrier arrive.
//   warp 1      MMA issuer     tcgen05.mma.cta_group::1.kind::f16, M = 128, N = N_TILE, K = 16, up to 4 per k-block
//                              (fewer on a ragged K tail), accumulating in TMEM (double-buffered: 2 x N_TILE columns);
//                              tcgen05.commit frees the A stage and the W stage.
//   warps 2-5   epilogue       tcgen05.ld -> + bias, ReLU6 -> bf16 -> swizzled staging panel -> cp.async.bulk.tensor.4d
//                              STORE of a [64 ch, TW, TH] box (the tensor map clips image edges and ragged N).
// The segment -> warp assignment is fixed for the whole kernel (no integer division in the loop).
#include <cuda.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "ptx.cuh"

namespace pn {

#ifndef PN_SEP_DW_WARPS
#define PN_SEP_DW_WARPS 10
#endif
constexpr int SEP_DW_WARPS = PN_SEP_DW_WARPS;
constexpr int SEP_FIRST_DW_WARP = 6;
constexpr int SEP_THREADS = (SEP_FIRST_DW_WARP + SEP_DW_WARPS) * 32;   // 512
constexpr int SEP_MAX_A = 6;
constexpr int SEP_A_BYTES = 128 * 128;                                 // 128 rows x 64 bf16
constexpr int SEP_STG_BYTES = 128 * 128;                               // one 128 x 64 bf16 output panel
constexpr int SEP_MAX_P = 6, SEP_MAX_W = 6;
constexpr int SEP_WGT_BYTES = 9 * 64 * 4 + 64 * 4;                     // dw weights [9][64] + bias [64] fp32
constexpr int SEP_SMEM_MAX = 232448;
constexpr int SEP_DWW_KB_BYTES = 10 * 64 * 4;                          // resident depthwise weights + bias of one k-block
constexpr unsigned SEP_EPI_SLEEP_NS = 200;                             // between the epilogue's polls of its accumulator barrier

struct SepGeom {
    int k, nc, ho, wo, pad;
    int th, tw, subs, ths, thi, twi;      // output tile, sub-tiles (rows per sub), input box
    int spr, seg_rows, segs_per_sub;      // 4-pixel column strips per tile row; rows per segment; segments per sub-tile
    unsigned segtab[64];                  // per segment: strip column | first output row << 8 | rows << 16 (rows are RSTEP apart)
    int tiles_x, tiles_y, n_tiles, n_tile, panels, tmem_cols;
    int n_halves, n_half, acc_bufs;       // a tile's accumulator = n_halves UMMA column blocks of n_half (<= 256) columns
    int kblocks;
    int half, cbox;                       // K <= 32: two pixel columns per warp (16 lanes each), 32-channel patch box
    int dww_res;                          // depthwise weights resident in shared memory (off_dww) instead of behind every patch stage
    int w_res;                            // pointwise weights resident: W stage = k-block * n_halves + column block, loaded once
    unsigned off_dww;                     // resident depthwise weights [kblocks][10][64] fp32 (SEP_LEAN & 4)
    int teams;                            // depthwise warp teams (1, 2): a team owns whole items, the teams take items in turn
    int p_stages, w_stages, a_stages, stg_bufs;
    unsigned patch_stage_bytes, patch_box_bytes, wgt_off, w_stage_bytes;
    unsigned off_a, off_stg, off_patch, off_bias, off_bar;   // from the 1024-aligned base; W stages sit at 0
    long long tiles;                      // m_tiles * n_tiles
};

struct SepBars {       // byte offsets of the mbarriers inside the barrier block
    static constexpr int patch_full = 0, patch_empty = 8 * SEP_MAX_P, w_full = 16 * SEP_MAX_P,
                         w_empty = 16 * SEP_MAX_P + 8 * SEP_MAX_W, a_full = 16 * SEP_MAX_P + 16 * SEP_MAX_W,
                         a_empty = a_full + 8 * SEP_MAX_A, tfull = a_empty + 8 * SEP_MAX_A, tempty = tfull + 16,
                         tmem_slot = tempty + 16, seg_ctr = tmem_slot + 16, seg_tab = seg_ctr + 4 * 8, total = seg_tab + 4 * 64;
};

__device__ __forceinline__ uint64_t sep_smem_desc(uint32_t saddr) {      // K-major SWIZZLE_128B (see gemm_tc.cu)
    return (uint64_t)((saddr & 0x3FFFF) >> 4) | (1ull << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
__device__ __forceinline__ uint32_t sep_idesc(int n) {                   // D f32, A/B bf16, K-major, M = 128
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}
__device__ __forceinline__ void sep_epi_bar() { asm volatile("bar.sync 1, 128;" ::: "memory"); }
__device__ __forceinline__ float4 lds_f4(uint32_t addr) {
    float4 r;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "r"(addr));
    return r;
}
__device__ __forceinline__ bool mbar_test(uint32_t bar, uint32_t parity) {             // non-blocking phase test
    uint32_t done;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    return done != 0;
}
__device__ __forceinline__ float2 lds_f2(uint32_t addr) {
    float2 r;
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(r.x), "=f"(r.y) : "r"(addr));
    return r;
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
    uint32_t r;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(r) : "r"(addr));
    return r;
}
__device__ __forceinline__ void sts_u32_if(uint32_t addr, uint32_t v, bool on) {     // compiles to one predicated STS; the predicate
    if (on) asm volatile("st.shared.b32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");  // is loop-invariant and stays in a P register
}

// Register window of the depthwise stencil for a strip of 4 output pixels: output row t reads input rows
// t*S + ky*D.  The window slides: a ring of NR rows, S new rows per step, PRE rows preloaded.  With dilation D > 1
// (stride 1) a segment walks the output rows of ONE residue class mod D (t, t+D, t+2D, ...): in that row space the
// stencil is dense again (rows t, t+D, t+2D -> one new row per step), so RSTEP = D scales the row pitch and the
// ring logic is the dilation-1 one (DR = 1).
// HALF (K <= 32 channels): lanes 0-15 own the even pixels of an 8-pixel strip, lanes 16-31 the odd ones, i.e. each lane
// walks 4 pixels that are HS = 2 S input columns apart -- no lane idles on zero-filled channels.
template <int S, int D, bool HALF> struct SepDwCfg {
    static constexpr bool SLIDE = true;
    static constexpr int RSTEP = (S == 1) ? D : 1;   // output / input row stride of a segment
    static constexpr int DR = (S == 1) ? 1 : D;      // row dilation in the segment's row space
    static constexpr bool UNPACKED = (D <= 2);       // window kept as fp32 pairs (18-27 pairs); wider windows stay packed
    static constexpr int NR = 2 * DR + 1;
    static constexpr int HS = HALF ? 2 * S : S;      // input columns between a lane's consecutive output pixels
    static constexpr int NCOLS = 3 * HS + 2 * D + 1;
    static constexpr int PRE = 2 * DR + 1 - S;
};


// Optional timeline trace (compile with -DPN_SEP_TRACE, see tools/trace_sep.py): block 0 stamps clock64 per role.
#ifdef PN_SEP_TRACE
__device__ long long *g_sep_trace = nullptr;
__device__ int g_sep_trace_cap = 0;
#endif
#if defined(PN_SEP_TRACE) && !defined(PN_SEP_PHASES)
#define SEP_TRACE(role, idx, what)                                                                               \
    do {                                                                                                         \
        if (blockIdx.x == 0 && g_sep_trace && (idx) < g_sep_trace_cap)                                           \
            g_sep_trace[((role) * g_sep_trace_cap + (idx)) * 4 + (what)] = clock64();                            \
    } while (0)
#else
#define SEP_TRACE(role, idx, what) do { } while (0)
#endif

// Phase timers of the depthwise warps (debug build: -DPN_SEP_TRACE -DPN_SEP_PHASES, tools/phases_sep.py): cycle sums per phase kept
// in registers (a clock read costs a few cycles, nothing goes to memory until the kernel ends), written by block 0 into the
// trace buffer, one row of 8 per depthwise warp: [wait A, wait patch, weights + table, window preload, rows, patch arrive,
// fence + A arrive, between items].
#ifdef PN_SEP_PHASES
#define SEP_PH_DECL long long ph_acc[8] = {0, 0, 0, 0, 0, 0, 0, 0}, ph_t = clock64()
#define SEP_PH(i) do { const long long ph_n = clock64(); ph_acc[i] += ph_n - ph_t; ph_t = ph_n; } while (0)
#else
#define SEP_PH_DECL do { } while (0)
#define SEP_PH(i) do { } while (0)
#endif

template <int S, int D, bool HALF>
__global__ void __launch_bounds__(SEP_THREADS, 1)
sepconv_kernel(const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_dww,
               const __grid_constant__ CUtensorMap tmap_dwb, const __grid_constant__ CUtensorMap tmap_w,
               const __grid_constant__ CUtensorMap tmap_y, const float *__restrict__ pw_bias, __nv_bfloat16 *__restrict__ y,
               const float *__restrict__ dw_w, const float *__restrict__ dw_b, const SepGeom g) {
    constexpr int CB = 64;                                  // channels per k-block (ragged K is zero-filled by TMA)
    const bool DWW_RES = g.dww_res != 0;                     // depthwise weights resident in shared memory (per block: sep_geometry)
    const long long tile_first = blockIdx.x, tile_step = gridDim.x;

    extern __shared__ uint8_t sep_smem_raw[];
    const uint32_t base = (smem_u32(sep_smem_raw) + 1023u) & ~1023u;
    const uint32_t bars = base + g.off_bar;
    auto bar = [&](int which, int s) { return bars + (uint32_t)which + 8u * (uint32_t)s; };
    auto w_addr = [&](int s) { return base + (uint32_t)s * g.w_stage_bytes; };
    auto a_addr = [&](int s) { return base + g.off_a + (uint32_t)s * SEP_A_BYTES; };
    auto p_addr = [&](int s) { return base + g.off_patch + (uint32_t)s * g.patch_stage_bytes; };
    volatile uint32_t *tmem_slot_ptr =
        reinterpret_cast<volatile uint32_t *>(sep_smem_raw + (base - smem_u32(sep_smem_raw)) + g.off_bar + SepBars::tmem_slot);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m_tiles_per_img = g.tiles_x * g.tiles_y;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmap_x);
        tma_prefetch_desc(&tmap_dww);
        tma_prefetch_desc(&tmap_dwb);
        tma_prefetch_desc(&tmap_w);
        tma_prefetch_desc(&tmap_y);
        for (int s = 0; s < g.p_stages; ++s) {
            mbar_init(bar(SepBars::patch_full, s), 1);
            mbar_init(bar(SepBars::patch_empty, s), SEP_DW_WARPS / g.teams);
        }
        for (int s = 0; s < g.w_stages; ++s) {
            mbar_init(bar(SepBars::w_full, s), 1);
            mbar_init(bar(SepBars::w_empty, s), 1);
        }
        for (int s = 0; s < g.a_stages; ++s) {
            mbar_init(bar(SepBars::a_full, s), SEP_DW_WARPS / g.teams);
            mbar_init(bar(SepBars::a_empty, s), 1);
        }
        for (int s = 0; s < 2; ++s) {
            mbar_init(bar(SepBars::tfull, s), 1);
            mbar_init(bar(SepBars::tempty, s), 128);
        }
        mbar_fence_init();
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(bars + (uint32_t)SepBars::tmem_slot),
                     "r"((uint32_t)g.tmem_cols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    {   // depthwise segment table (strip column | first row << 8 | rows << 16)
        uint32_t *misc = reinterpret_cast<uint32_t *>(sep_smem_raw + (base - smem_u32(sep_smem_raw)) + g.off_bar);
        if ((int)threadIdx.x < g.segs_per_sub) misc[SepBars::seg_tab / 4 + threadIdx.x] = g.segtab[threadIdx.x];
    }
    {   // pointwise bias -> shared memory once (the epilogue reads it per panel)
        float *sbias = reinterpret_cast<float *>(sep_smem_raw + (base - smem_u32(sep_smem_raw)) + g.off_bias);
        const int ncp = g.n_tiles * g.panels * 64;                // padded so that ragged panels read zeros
        for (int i = threadIdx.x; i < ncp; i += SEP_THREADS) sbias[i] = i < g.nc ? __ldg(pw_bias + i) : 0.f;
    }
    if (DWW_RES) {   // depthwise weights [9, K] + bias [K] -> [k-block][tap | bias][64] fp32, ragged K zero-filled (never written by the
                     // preceding kernel, so this may run before griddepcontrol.wait like the bias above)
        float *sw = reinterpret_cast<float *>(sep_smem_raw + (base - smem_u32(sep_smem_raw)) + g.off_dww);
        for (int i = threadIdx.x; i < g.kblocks * 640; i += SEP_THREADS) {
            const int kbi = i / 640, r = i - kbi * 640, t = r >> 6, ch = kbi * 64 + (r & 63);
            sw[i] = ch < g.k ? (t < 9 ? __ldg(dw_w + (size_t)t * g.k + ch) : __ldg(dw_b + ch)) : 0.f;
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    pdl_launch_dependents();                                  // after the TMEM allocation is made (see stem.cu): a dependent CTA must not allocate first
    pdl_wait();                                               // everything above overlapped the previous layer's tail
    const uint32_t tmem_base = *tmem_slot_ptr;

    if (warp == 0) {
        // ===================== TMA producer =====================
        // One thread feeds two independent rings -- input patches (+ depthwise weights) and pointwise weight blocks --
        // each with its own cursor over (tile, k-block, ...), polled without blocking so that a full W ring never holds
        // back a patch load (the depthwise warps run ahead of the MMA by the depth of the A ring).
        if (lane == 0) {
            int ps = 0, ws = 0, tr_p = 0;
            uint32_t pph = 0, wph = 0;
            (void)tr_p;
            long long p_tile = tile_first, w_tile = tile_first;
            int p_kb = 0, p_sub = 0, w_kb = 0, w_hf = 0;
            int p_img = 0, p_ty = 0, p_tx = 0, w_col = 0;
            bool p_new = true, w_new = true;
            const long long t0 = clock64();
            while (p_tile < g.tiles || w_tile < g.tiles) {
                bool progress = false;
                if (p_tile < g.tiles) {
                    if (p_new) {
                        const int m_tile = (int)(p_tile / g.n_tiles);
                        p_img = m_tile / m_tiles_per_img;
                        const int rem = m_tile - p_img * m_tiles_per_img;
                        p_ty = rem / g.tiles_x;
                        p_tx = rem - p_ty * g.tiles_x;
                        p_new = false;
                    }
                    if (mbar_test(bar(SepBars::patch_empty, ps), pph ^ 1)) {
                        const uint32_t full = bar(SepBars::patch_full, ps);
                        SEP_TRACE(3, tr_p, 0);
                        mbar_expect_tx(full, g.patch_box_bytes + (DWW_RES ? 0u : (uint32_t)SEP_WGT_BYTES));
                        tma_load_4d(p_addr(ps), &tmap_x, full, p_kb * CB, p_tx * g.tw * S - g.pad,
                                    (p_ty * g.th + p_sub * g.ths) * S - g.pad, p_img);
                        if (!DWW_RES) {
                            tma_load_2d(p_addr(ps) + g.wgt_off, &tmap_dww, full, p_kb * CB, 0);
                            tma_load_2d(p_addr(ps) + g.wgt_off + 9 * 64 * 4, &tmap_dwb, full, p_kb * CB, 0);
                        }
                        SEP_TRACE(3, tr_p, 1);
                        ++tr_p;
                        if (++ps == g.p_stages) { ps = 0; pph ^= 1; }
                        if (++p_sub == g.subs) {
                            p_sub = 0;
                            if (++p_kb >= g.kblocks) { p_kb = 0; p_tile += tile_step; p_new = true; }
                        }
                        progress = true;
                    }
                }
                if (w_tile < g.tiles) {
                    if (w_new) { w_col = (int)(w_tile % g.n_tiles) * g.n_tile; w_new = false; }
                    if (mbar_test(bar(SepBars::w_empty, ws), wph ^ 1)) {
                        mbar_expect_tx(bar(SepBars::w_full, ws), g.w_stage_bytes);
                        tma_load_2d(w_addr(ws), &tmap_w, bar(SepBars::w_full, ws), w_kb * CB, w_col + w_hf * g.n_half);
                        if (++ws == g.w_stages) { ws = 0; wph ^= 1; }
                        if (++w_hf == g.n_halves) {
                            w_hf = 0;
                            if (++w_kb == g.kblocks) {
                                w_kb = 0; w_tile += tile_step; w_new = true;
                                if (g.w_res) w_tile = g.tiles;          // resident W: every (k-block, column block) has its own stage, loaded once
                            }
                        }
                        progress = true;
                    }
                }
                if (!progress) {
                    __nanosleep(32);                                   // nothing to refill: leave the issue slots to the depthwise warps
                    if (clock64() - t0 > 20000000000ll) {              // ~10 s: a protocol bug, never a slow kernel
                        printf("posenet_b200: sepconv producer timeout (block %d)\n", blockIdx.x);
                        __trap();
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        if (lane == 0) {
            const uint32_t idesc = sep_idesc(g.n_half);
            int as = 0, ws = 0, acc = 0, tr_i = 0;
            uint32_t aph = 0, wph = 0, acc_phase = 0;
            (void)tr_i;
            for (long long tile = tile_first; tile < g.tiles; tile += tile_step) {
                mbar_wait(bar(SepBars::tempty, acc), acc_phase ^ 1);
                tc_fence_after();
                SEP_TRACE(1, tr_i, 0);
                const uint32_t d_tmem = tmem_base + (uint32_t)(acc * g.n_tile);
                for (int kb = 0; kb < g.kblocks; ++kb) {
                    mbar_wait(bar(SepBars::a_full, as), aph);
                    SEP_TRACE(1, tr_i, 1);
                    const uint32_t sa = a_addr(as);
                    const int rem_k = g.k - kb * CB;                             // ragged K tail: only the k16 steps that hold channels
                    const int ksteps = rem_k >= CB ? CB / 16 : (rem_k + 15) / 16;
                    for (int hf = 0; hf < g.n_halves; ++hf) {
                        if (g.w_res) {                                // resident W: stage = (k-block, column block); landed once, in phase 0
                            ws = kb * g.n_halves + hf;
                            if (tile == tile_first) mbar_wait(bar(SepBars::w_full, ws), 0);
                        } else
                            mbar_wait(bar(SepBars::w_full, ws), wph);
                        tc_fence_after();
                        const uint32_t sb = w_addr(ws);
#pragma unroll
                        for (int k = 0; k < CB / 16; ++k)
                            if (k < ksteps)
                                tc_mma_bf16(d_tmem + (uint32_t)(hf * g.n_half), sep_smem_desc(sa + k * 32), sep_smem_desc(sb + k * 32), idesc,
                                            (uint32_t)((kb | k) != 0));
                        if (!g.w_res) {
                            tc_commit(bar(SepBars::w_empty, ws));
                            if (++ws == g.w_stages) { ws = 0; wph ^= 1; }
                        }
                    }
                    tc_commit(bar(SepBars::a_empty, as));
                    SEP_TRACE(1, tr_i, 2);
                    ++tr_i;
                    if (++as == g.a_stages) { as = 0; aph ^= 1; }
                }
                tc_commit(bar(SepBars::tfull, acc));
                if (++acc == g.acc_bufs) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else if (warp < SEP_FIRST_DW_WARP) {
        // ===================== epilogue (warps 2..5) =====================
        const int q = warp & 3;                                          // TMEM lane quarter this warp may read
        const int row_in_tile = q * 32 + lane;
        const bool issuer = (threadIdx.x == 64);
        const uint32_t staging = base + g.off_stg;
        int acc = 0, buf = 0, tr_e = 0;
        uint32_t acc_phase = 0;
        (void)tr_e;
        if (g.stg_bufs == 0) {
            // ---- direct epilogue: TMEM -> registers -> global, no staging panel, no CTA-level barrier.  A thread owns one tile row
            // (= one output pixel): 32 accumulator columns are 64 contiguous bytes of its NHWC pixel, written as two 32-byte
            // stores (whole sectors).  The tcgen05.ld of chunk c + 1 is in flight while chunk c is converted and stored.
            const int r_ty = row_in_tile / g.tw, r_tx = row_in_tile - r_ty * g.tw;
            const int chunks = (g.n_tile + 31) >> 5;
            auto emit = [&](const uint32_t (&v)[32], int c, __nv_bfloat16 *yrow, bool row_ok, int col_lim, uint32_t bias_base) {
                const int col0 = c * 32;                                  // column inside this tile's n_tile block
#pragma unroll
                for (int piece = 0; piece < 2; ++piece) {
                    uint32_t o[8];
#pragma unroll
                    for (int j = 0; j < 8; j += 2) {
                        const float4 b0 = lds_f4(bias_base + (uint32_t)(col0 + piece * 16 + j * 2) * 4u);
                        const int i0 = piece * 16 + j * 2;
                        const float2 s0 = fadd2(make_float2(__uint_as_float(v[i0 + 0]), __uint_as_float(v[i0 + 1])), make_float2(b0.x, b0.y));
                        const float2 s1 = fadd2(make_float2(__uint_as_float(v[i0 + 2]), __uint_as_float(v[i0 + 3])), make_float2(b0.z, b0.w));
                        o[j] = relu6_bf16x2(s0);
                        o[j + 1] = relu6_bf16x2(s1);
                    }
                    if (row_ok && col0 + piece * 16 < col_lim)
                        asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(yrow + col0 + piece * 16), "r"(o[0]),
                                     "r"(o[1]), "r"(o[2]), "r"(o[3]), "r"(o[4]), "r"(o[5]), "r"(o[6]), "r"(o[7])
                                     : "memory");
                }
            };
            for (long long tile = tile_first; tile < g.tiles; tile += tile_step) {
                const int n_tile = (int)(tile % g.n_tiles);
                const int m_tile = (int)(tile / g.n_tiles);
                const int img = m_tile / m_tiles_per_img;
                const int rem = m_tile - img * m_tiles_per_img;
                const int ty = rem / g.tiles_x, tx = rem - ty * g.tiles_x;
                const int oy = ty * g.th + r_ty, ox = tx * g.tw + r_tx;
                const bool row_ok = r_ty < g.th && oy < g.ho && ox < g.wo;
                const int colg = n_tile * g.n_tile;                       // first output channel of this accumulator
                __nv_bfloat16 *yrow = y + (((size_t)img * g.ho + oy) * g.wo + ox) * (size_t)g.nc + colg;
                const int col_lim = g.nc - colg;                          // columns of this block that exist (ragged N)
                mbar_wait_backoff(bar(SepBars::tfull, acc), acc_phase, SEP_EPI_SLEEP_NS);
                tc_fence_after();
                if (issuer) SEP_TRACE(2, tr_e, 0);
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * g.n_tile);
                const uint32_t bias_base = base + g.off_bias + (uint32_t)(n_tile * g.n_tile) * 4u;   // this block's bias in shared memory
                uint32_t va[32], vb[32];
                tc_ld32(taddr, va);
#pragma unroll 1
                for (int c = 0; c < chunks; c += 2) {
                    tc_ld_wait();
                    if (c + 1 < chunks) tc_ld32(taddr + (uint32_t)((c + 1) * 32), vb);
                    else { tc_fence_before(); mbar_arrive(bar(SepBars::tempty, acc)); }
                    emit(va, c, yrow, row_ok, col_lim, bias_base);
                    if (c + 1 < chunks) {
                        tc_ld_wait();
                        if (c + 2 < chunks) tc_ld32(taddr + (uint32_t)((c + 2) * 32), va);
                        else { tc_fence_before(); mbar_arrive(bar(SepBars::tempty, acc)); }
                        emit(vb, c + 1, yrow, row_ok, col_lim, bias_base);
                    }
                }
                if (issuer) { SEP_TRACE(2, tr_e, 1); ++tr_e; }
                if (++acc == g.acc_bufs) { acc = 0; acc_phase ^= 1; }
            }
        } else
        for (long long tile = tile_first; tile < g.tiles; tile += tile_step) {
            const int n_tile = (int)(tile % g.n_tiles);
            const int m_tile = (int)(tile / g.n_tiles);
            const int img = m_tile / m_tiles_per_img;
            const int rem = m_tile - img * m_tiles_per_img;
            const int ty = rem / g.tiles_x, tx = rem - ty * g.tiles_x;
            mbar_wait_backoff(bar(SepBars::tfull, acc), acc_phase, SEP_EPI_SLEEP_NS);   // idle epilogue warps must not eat issue slots
            tc_fence_after();
            if (issuer) SEP_TRACE(2, tr_e, 0);
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * g.n_tile);
#pragma unroll 1
            for (int p = 0; p < g.panels; ++p) {
                const int col0 = n_tile * g.n_tile + p * 64;
                if (issuer) {                                            // the store that last read this buffer is done
                    if (g.stg_bufs == 2) bulk_wait_read<1>(); else bulk_wait_read<0>();
                }
                sep_epi_bar();
                const uint32_t srow = staging + (uint32_t)buf * SEP_STG_BYTES + (uint32_t)row_in_tile * 128u;
#pragma unroll
                for (int hf = 0; hf < 2; ++hf) {
                    uint32_t v[32];
                    tc_ld32(taddr + (uint32_t)(p * 64 + hf * 32), v);
                    tc_ld_wait();
                    if (p == g.panels - 1 && hf == 1) {                  // accumulator fully in registers: hand it back
                        tc_fence_before();
                        mbar_arrive(bar(SepBars::tempty, acc));
                    }
#pragma unroll
                    for (int c = 0; c < 4; ++c) {                        // 8 columns -> one 16 B chunk, 128B-swizzled
                        const uint32_t bsm = base + g.off_bias + (uint32_t)(col0 + hf * 32 + c * 8) * 4u;
                        const float4 b0 = lds_f4(bsm), b1 = lds_f4(bsm + 16);
                        const float2 s0 = fadd2(make_float2(__uint_as_float(v[8 * c + 0]), __uint_as_float(v[8 * c + 1])), make_float2(b0.x, b0.y));
                        const float2 s1 = fadd2(make_float2(__uint_as_float(v[8 * c + 2]), __uint_as_float(v[8 * c + 3])), make_float2(b0.z, b0.w));
                        const float2 s2 = fadd2(make_float2(__uint_as_float(v[8 * c + 4]), __uint_as_float(v[8 * c + 5])), make_float2(b1.x, b1.y));
                        const float2 s3 = fadd2(make_float2(__uint_as_float(v[8 * c + 6]), __uint_as_float(v[8 * c + 7])), make_float2(b1.z, b1.w));
                        st_shared_v4(srow + (uint32_t)(((hf * 4 + c) ^ (row_in_tile & 7)) << 4), relu6_bf16x2(s0), relu6_bf16x2(s1),
                                     relu6_bf16x2(s2), relu6_bf16x2(s3));
                    }
                }
                fence_async_smem();                                      // generic writes -> visible to TMA
                sep_epi_bar();
                if (issuer) {
                    tma_store_4d(&tmap_y, staging + (uint32_t)buf * SEP_STG_BYTES, col0, tx * g.tw, ty * g.th, img);
                    bulk_commit();
                }
                if (g.stg_bufs == 2) buf ^= 1;
            }
            if (issuer) { SEP_TRACE(2, tr_e, 1); ++tr_e; }
            if (++acc == g.acc_bufs) { acc = 0; acc_phase ^= 1; }
        }
        if (issuer) bulk_wait_all();                                     // smem must outlive the last bulk store
    } else {
        // ===================== depthwise producers of the A tile (warps 6..15) =====================
        // Lane l owns channels 2l, 2l+1 of the 64-channel k-block (4 B of every pixel).  A warp takes the next segment --
        // a column strip of 4 output pixels (8 when HALF) x up to seg_rows rows of one (tile, k-block, sub-tile) item --
        // from the CTA-wide counter, and slides down its rows keeping the input-row window of the 3x3 stencil in registers
        // (fp32 pairs for dilation 1, bf16 pairs otherwise), so every patch element is read from shared memory once per
        // segment, unpacked once, and the 9 x 2 weights + bias stay in registers for the segment.  The rows entering the
        // window at the next step are prefetched before the FMAs of the current one.  One ld.shared.b32 / st.shared.b32
        // is one conflict-free 128 B wavefront per warp.  Items are handed out in order, so a warp that finishes early
        // simply starts on the next item's patch (if it has landed) while the others complete the current A stage.
        using Cfg = SepDwCfg<S, D, HALF>;
        constexpr int NR = Cfg::NR, NCOLS = Cfg::NCOLS, PRE = Cfg::PRE, HS = Cfg::HS, RSTEP = Cfg::RSTEP, DR = Cfg::DR;
        constexpr bool SLIDE = Cfg::SLIDE, UNPACKED = Cfg::UNPACKED, PREFETCH = Cfg::UNPACKED;
        constexpr int NNEW = S;                                      // input rows loaded per step
        constexpr uint32_t PIX = HALF ? 64u : 128u;                  // bytes per patch pixel
        const int hsel = HALF ? (lane >> 4) : 0, cp = HALF ? (lane & 15) : lane;
        const uint32_t rowb1 = (uint32_t)g.twi * PIX, rowb = rowb1 * RSTEP;      // patch row pitch; pitch between a segment's rows
        const uint32_t lane_off = (uint32_t)(hsel * S) * PIX + (uint32_t)cp * 4u;
        const uint32_t a_lane = (uint32_t)(cp >> 2) << 4 | (uint32_t)(cp & 3) << 2;       // 16 B chunk | byte inside it
        auto unpack = [](uint32_t r) { return make_float2(__uint_as_float(r << 16), __uint_as_float(r & 0xffff0000u)); };
        const uint32_t tab_addr = bars + (uint32_t)SepBars::seg_tab;

        // Every warp walks all items -- (tile, k-block, sub-tile), one patch stage each -- in order, so its mbarrier parities
        // never skip a phase.  Inside an item the segments are assigned statically: warp w takes segments (w + item) mod
        // DW_WARPS, + DW_WARPS, ... -- the rotation spreads the short segments (and the warp left without one when there are
        // 9 segments for 10 warps) over all warps and schedulers.  A shared-memory counter handing the segments out on demand
        // balanced an item a little better but cost an atomic, a shuffle and two divergent branches per grab, i.e. 10-15 % of
        // a depthwise warp's time at one ~2000-cycle segment per warp and item (ncu source view: `branch_resolving` and
        // `short_scoreboard` on the grab, 6 % of the kernel on four shapes).  A warp without work in an item moves straight on
        // to the next one while the others finish.
        //
        // Teams (g.teams == 2): the hand-off protocol of an item -- two mbarrier probes, the proxy fence, two arrives, the weight
        // loads: ~1.5k cycles of fixed round trips through the shared-memory unit against ~1.4k cycles of stencil work per
        // warp (tools/phases_sep.py) -- is paid by every warp that takes part in the item.  So the ten warps form two teams of
        // five that own WHOLE items, even items one team, odd items the other: a warp does two segments per hand-off instead
        // of one, the barriers count five arrivals, and two items are in flight at once (the rings are deep enough where
        // sep_geometry turns this on).  Every warp still walks all items in order so that its stage cursors and parities
        // follow the rings; it just steps over the other team's items.
        const int n_teams = g.teams, dwi = warp - SEP_FIRST_DW_WARP, team_warps = SEP_DW_WARPS / n_teams;
        const int team = dwi / team_warps, team_first = team * team_warps;
        const int n_subs = g.subs, n_pst = g.p_stages, n_ast = g.a_stages, n_kb = g.kblocks;
        int tr_d = 0;
        // cursors of this warp's first item, item `team` (its stages follow the first team's: both rings are deeper than one item)
        int ps = team * n_subs, as = team, kb = team;
        uint32_t pph = 0, aph = 0;
        int rot = dwi - team_first;                                      // this warp's first segment in the current item
        long long tile = tile_first;
        while (kb >= n_kb) { kb -= n_kb; tile += tile_step; }              // (single-k-block tiles: the second team starts one tile on)
        (void)tr_d;
        const bool tracer = (warp == SEP_FIRST_DW_WARP && lane == 0);
        (void)tracer;
        SEP_PH_DECL;
        float2 wk[9], bias2;                                          // this lane's 9 taps + bias of its channel pair
        int wk_kb = -1;                                               // DWW_RES: k-block whose weights the registers hold
        (void)wk_kb;
        while (tile < g.tiles) {
          {
            SEP_PH(7);
            if (tracer) SEP_TRACE(0, tr_d, 0);
            if (DWW_RES && kb != wk_kb) {
                // resident weights: requested BEFORE the barrier probe so that the two shared-memory round trips overlap; a warp
                // that keeps its k-block from item to item (k-blocks == teams) loads them once per kernel
                const uint32_t wsm = base + g.off_dww + (uint32_t)kb * (uint32_t)SEP_DWW_KB_BYTES + (uint32_t)cp * 8u;
#pragma unroll
                for (int t = 0; t < 9; ++t) wk[t] = lds_f2(wsm + (uint32_t)t * 256u);
                bias2 = lds_f2(wsm + 9 * 256u);
                wk_kb = kb;
            }
            mbar_wait(bar(SepBars::a_empty, as), aph ^ 1);            // the MMAs that read this A stage have retired
            if (tracer) SEP_TRACE(0, tr_d, 1);
            SEP_PH(0);
            const uint32_t a_stage = a_addr(as);
            for (int sub = 0; sub < n_subs; ++sub) {
              mbar_wait(bar(SepBars::patch_full, ps), pph);
              if (tracer && sub == 0) SEP_TRACE(0, tr_d, 2);
              SEP_PH(1);
              const uint32_t stage = p_addr(ps);
              bool have_w = DWW_RES;
              for (int seg = rot; seg < g.segs_per_sub; seg += team_warps) {
                if (!have_w) {
                    const uint32_t wsm = stage + g.wgt_off + (uint32_t)cp * 8u;
#pragma unroll
                    for (int t = 0; t < 9; ++t) wk[t] = lds_f2(wsm + (uint32_t)t * 256u);
                    bias2 = lds_f2(wsm + 9 * 256u);
                    have_w = true;
                }
                const uint32_t tab = lds_u32(tab_addr + (uint32_t)seg * 4u);
                const int s_col = (int)(tab & 0xffu), s_r0 = (int)((tab >> 8) & 0xffu), s_n = (int)(tab >> 16);
                const int orow0 = sub * g.ths + s_r0;
                const int nrows = min(s_n, (g.th - orow0 + RSTEP - 1) / RSTEP);     // rows of this segment inside the tile
                SEP_PH(2);
                if (nrows > 0) {
                    const uint32_t src = stage + (uint32_t)(s_r0 * S) * rowb1 + (uint32_t)(s_col * S) * PIX + lane_off;
                    const int ncol_ok = g.tw - s_col;                               // strip pixels px < ncol_ok exist
                    int arow = orow0 * g.tw + s_col;                                // A-tile row == TMEM lane == staging row

                    float2 ringf[UNPACKED ? NR : 1][NCOLS];                         // the window, unpacked (dilation 1)
                    uint32_t ringp[UNPACKED ? 1 : NR][NCOLS];                       // ... or packed bf16 pairs
                    uint32_t nxt[PREFETCH ? NNEW : 1][NCOLS];                       // rows entering the window next
                    if (SLIDE) {
    #pragma unroll
                        for (int r = 0; r < PRE; ++r)
    #pragma unroll
                            for (int c = 0; c < NCOLS; ++c) {
                                const uint32_t v = lds_u32(src + (uint32_t)r * rowb + (uint32_t)c * PIX);
                                if (UNPACKED) ringf[r][c] = unpack(v); else ringp[r][c] = v;
                            }
                        if (PREFETCH) {
    #pragma unroll
                            for (int n = 0; n < S; ++n)
    #pragma unroll
                                for (int c = 0; c < NCOLS; ++c) nxt[n][c] = lds_u32(src + (uint32_t)(PRE + n) * rowb + (uint32_t)c * PIX);
                        }
                    }
                    SEP_PH(3);
    #pragma unroll 1
                    for (int t0 = 0; t0 < nrows; t0 += NR) {
    #pragma unroll
                        for (int j = 0; j < NR; ++j) {
                            const int t = t0 + j;
                            if (t >= nrows) break;
                            if (PREFETCH) {
                                // the prefetched rows enter the window ...
    #pragma unroll
                                for (int n = 0; n < NNEW; ++n)
    #pragma unroll
                                    for (int c = 0; c < NCOLS; ++c) {
                                        const int slot = (PRE + j * S + n) % NR;
                                        if (UNPACKED) ringf[slot][c] = unpack(nxt[n][c]); else ringp[slot][c] = nxt[n][c];
                                    }
                                // ... and the next step's rows are requested before this step's math.  After the last row the
                                // request repeats the last one (a predicated load would cost a register copy per element)
                                {
                                    const int tn = t + 1 < nrows ? t + 1 : t;
    #pragma unroll
                                    for (int n = 0; n < NNEW; ++n) {
                                        const uint32_t rp = src + (uint32_t)(PRE + tn * S + n) * rowb;
    #pragma unroll
                                        for (int c = 0; c < NCOLS; ++c) nxt[n][c] = lds_u32(rp + (uint32_t)c * PIX);
                                    }
                                }
                            } else {
    #pragma unroll
                                for (int n = 0; n < NNEW; ++n) {
                                    const int slot = (PRE + j * S + n) % NR;
                                    const uint32_t rp = src + (uint32_t)(PRE + t * S + n) * rowb;
    #pragma unroll
                                    for (int c = 0; c < NCOLS; ++c) ringp[slot][c] = lds_u32(rp + (uint32_t)c * PIX);
                                }
                            }
                            float2 acc[4] = {bias2, bias2, bias2, bias2};
    #pragma unroll
                            for (int ky = 0; ky < 3; ++ky) {
                                const int slot = (j * S + ky * DR) % NR;
    #pragma unroll
                                for (int c = 0; c < NCOLS; ++c) {
                                    const float2 v = UNPACKED ? ringf[slot][c] : unpack(ringp[slot][c]);
    #pragma unroll
                                    for (int p = 0; p < 4; ++p)
    #pragma unroll
                                        for (int kx = 0; kx < 3; ++kx)
                                            if (p * HS + kx * D == c) acc[p] = ffma2(v, wk[ky * 3 + kx], acc[p]);
                                }
                            }
    #pragma unroll
                            for (int p = 0; p < 4; ++p) {
                                const int px = HALF ? 2 * p + hsel : p;                  // pixel inside the strip
                                const uint32_t r = (uint32_t)(arow + px);
                                sts_u32_if(a_stage + ((r << 7) | a_lane) ^ ((r & 7u) << 4), relu6_bf16x2(acc[p]), px < ncol_ok);
                            }
                            arow += g.tw * RSTEP;
                        }
                    }
                }
                SEP_PH(4);
              }   // segments of this item
              __syncwarp();
              if (lane == 0) mbar_arrive(bar(SepBars::patch_empty, ps));     // this warp no longer reads the patch
              SEP_PH(5);
              if (++ps == n_pst) { ps = 0; pph ^= 1; }
              if (++rot == team_warps) rot = 0;
            }
            fence_async_smem();                                       // A-tile writes -> visible to the tensor core
            __syncwarp();
            if (lane == 0) mbar_arrive(bar(SepBars::a_full, as));
            SEP_PH(6);
            if (tracer) { SEP_TRACE(0, tr_d, 3); ++tr_d; }
            // on to this warp's next item: over the other team's patch stages and A stage, n_teams k-blocks ahead
            if (n_teams > 1) {
                ps += (n_teams - 1) * n_subs;
                if (ps >= n_pst) { ps -= n_pst; pph ^= 1; }
            }
            as += n_teams;
            if (as >= n_ast) { as -= n_ast; aph ^= 1; }
            kb += n_teams;
            while (kb >= n_kb) { kb -= n_kb; tile += tile_step; }
          }
        }
#ifdef PN_SEP_PHASES
        if (blockIdx.x == 0 && lane == 0 && g_sep_trace && warp - SEP_FIRST_DW_WARP < g_sep_trace_cap)
            for (int i = 0; i < 8; ++i) g_sep_trace[(warp - SEP_FIRST_DW_WARP) * 8 + i] = ph_acc[i];
#endif
    }


    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)g.tmem_cols) : "memory");
    }
}

// ---- host side ---------------------------------------------------------------------------------------------
struct SepTuned { int k, nc, stride, dil, ho, wo, th, tw, subs, p, w, a, stg, teams; };
static const SepTuned SEP_TUNED[] = {
#include "sep_tuned.inc"
    {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0}};
static int next_pow2_cols(int c) {
    int p = 32;
    while (p < c) p <<= 1;
    return p;
}

bool sep_supported(int k, int nc, int stride, int dil) {
    return k % 8 == 0 && nc % 16 == 0 && k >= 8 && nc >= 16 &&
           ((stride == 1 && (dil == 1 || dil == 2 || dil == 4)) || (stride == 2 && dil == 1));
}

// Blocks worth running fused: whole output width in one accumulator tile (<= 512 channels); anything wider would redo the
// depthwise work once per 512 outputs and is faster as two kernels.
bool sep_fuse_recommended(int k, int nc, int stride, int dil) { return sep_supported(k, nc, stride, dil) && nc <= 512; }

// Tile shape, stage counts and the shared-memory carve-up for one block (pure host arithmetic, no CUDA calls).
int sep_geometry(SepOp *op, int n, int h, int wd, int k, int nc, int stride, int dil) {
    PN_CHECK_ARG(n > 0 && h > 0 && wd > 0, "pn_sepconv_block: bad shape");
    PN_CHECK_ARG(sep_supported(k, nc, stride, dil), "pn_sepconv_block: unsupported block (cin %d cout %d stride %d dilation %d)", k,
                 nc, stride, dil);
    memset(op, 0, sizeof(*op));
    if (sepwarp_supported(k, nc, stride, dil)) {                    // narrow block: warp-autonomous kernel, no tile geometry
        op->warp_kind = true;
        op->stride = stride; op->dil = dil;
        op->ho = (h - 1) / stride + 1; op->wo = (wd - 1) / stride + 1;
        op->n = n; op->h = h; op->w = wd; op->k = k; op->nc = nc;
        return PN_OK;
    }
    if (septc_supported(k, nc, stride, dil)) {                      // depthwise on the tensor pipe (septc.cu)
        op->tc_kind = true;
        op->stride = stride; op->dil = dil;
        op->ho = h; op->wo = wd;
        op->n = n; op->h = h; op->w = wd; op->k = k; op->nc = nc;
        return septc_geometry(&op->tc, n, h, wd, k, nc, dil);
    }
    SepGeom g;
    memset(&g, 0, sizeof(g));
    g.k = k; g.nc = nc;
    g.pad = ((stride - 1) + dil * 2) / 2;
    g.ho = (h + 2 * g.pad - 2 * dil - 1) / stride + 1;
    g.wo = (wd + 2 * g.pad - 2 * dil - 1) / stride + 1;
    PN_CHECK_ARG(g.ho > 0 && g.wo > 0, "pn_sepconv_block: empty output");
    const int cb = 64;
    const bool slide = dil == 1;
    // K <= 32 (the first block of every model): half-warp per pixel column, 32-channel patch box (sepconv_kernel HALF)
    g.half = (k <= 32 && stride == 1 && dil == 1) ? 1 : 0;
    g.cbox = g.half ? 32 : cb;
    const int sw = g.half ? 8 : 4;                                  // output pixels per strip step
    const int ncols = 3 * stride * (g.half ? 2 : 1) + 2 * dil + 1, pre = slide ? 2 * dil + 1 - stride : 0;
    g.kblocks = ceil_div(k, cb);
    // Output columns per tile: up to 256 double-buffered in TMEM (the epilogue of tile i overlaps the main loop of tile
    // i+1), or up to 512 as two UMMA column blocks single-buffered -- the depthwise work, which bounds the deep layers,
    // is then done once per 512 output channels instead of once per 256.
    g.n_tiles = ceil_div(nc, 512);
    g.n_tile = nc / g.n_tiles;
    g.n_halves = g.n_tile > 256 ? 2 : 1;                            // W ring granularity: UMMA column blocks of n_tile / n_halves columns
    g.n_half = g.n_tile / g.n_halves;
    PN_CHECK_ARG(g.n_tile * g.n_tiles == nc && g.n_half * g.n_halves == g.n_tile && g.n_half % 16 == 0,
                 "pn_sepconv_block: cout %d does not split into tiles", nc);
    g.panels = ceil_div(g.n_tile, 64);
    g.acc_bufs = g.n_tile > 256 ? 1 : 2;
    g.tmem_cols = g.n_tile > 256 ? 512 : next_pow2_cols(g.n_tile + g.panels * 64);
    PN_CHECK_ARG(g.tmem_cols <= 512 && g.panels * 64 <= 512, "pn_sepconv_block: TMEM budget exceeded");
    g.w_stage_bytes = (unsigned)g.n_half * 128u;

    // ---- resident weights.  Depthwise: [k-block][9 taps + bias][64] fp32 loaded once per kernel instead of
    // travelling behind every patch stage (K <= 256; beyond that 15-20 KB resident would cost a patch stage); a warp fetches its
    // registers from there while it probes the patch barrier.  Pointwise: where every (k-block, column block) fits a stage of its
    // own (<= 80 KB in all) the W ring is loaded once and never again -- per tile that is as much L2 -> shared-memory traffic as
    // the patches themselves, and the MMA thread loses a wait and a commit per k-block.  Measured on B200 (same tiles):
    // 128 -> 256 s2 @129^2 100.0 -> 96.2 us, 192 -> 192 @33^2 x512 135.7 -> 134.0, 128 -> 256 @91x161 114.8 -> 110.0; the freed
    // stages matter more where they buy a deeper ring or a larger tile.
    const bool dww_res = g.kblocks <= 4;
    const int wgt_stage = dww_res ? 0 : SEP_WGT_BYTES;             // depthwise weight bytes behind each patch stage
    const int dww_bytes = dww_res ? g.kblocks * SEP_DWW_KB_BYTES : 0;
    g.dww_res = dww_res ? 1 : 0;
    g.w_res = (g.n_tiles == 1 && g.kblocks * g.n_halves <= SEP_MAX_W &&
               (long long)g.kblocks * g.n_halves * g.w_stage_bytes <= 80 * 1024) ? 1 : 0;
    // ---- tile search: fewest (tiles x per-tile cost); one strip per depthwise thread group per sub-tile
    const int min_w = g.w_res ? g.kblocks * g.n_halves : g.n_halves >= 2 ? 3 : 2;   // default W ring entries (column blocks of a k-block, plus one ahead)
    const int fixed = 2 * SEP_A_BYTES + SEP_STG_BYTES + min_w * (int)g.w_stage_bytes + 1024 + 640 + 4224 + dww_bytes;   // minimum non-patch smem
    double best = 1e300;
    // Measured choices first (sep_tuned.inc: tools/tune_sep.py timed the tile shapes / ring depths of the blocks of the reference's
    // standard resolutions on a B200; the cost model below ranks them poorly -- up to 25 % between tiles it scores alike), the
    // model for every other shape.  PN_SEP_TILE="th,tw,subs" / PN_SEP_STAGES / PN_SEP_TEAMS force a choice (tools/tune_sep.py).
    const SepTuned *tuned = nullptr;
    for (const SepTuned &t : SEP_TUNED)
        if (t.k == k && t.nc == nc && t.stride == stride && t.dil == dil && t.ho == g.ho && t.wo == g.wo) { tuned = &t; break; }
    int f_th = 0, f_tw = 0, f_subs = 0;
    if (tuned) { f_th = tuned->th; f_tw = tuned->tw; f_subs = tuned->subs; }
    if (const char *force = getenv("PN_SEP_TILE"))
        if (sscanf(force, "%d,%d,%d", &f_th, &f_tw, &f_subs) != 3) f_th = f_tw = f_subs = 0;
    for (int th = 1; th <= 64; ++th) {
        for (int tw = 1; tw <= 64; ++tw) {
            if (th * tw > 128) break;
            if ((th - 1) >= g.ho + 7 || (tw - 1) >= g.wo + 7) continue;
            for (int subs = 1; subs <= 4 && subs <= th; ++subs) {
                if (f_th && (th != f_th || tw != f_tw || subs != f_subs)) continue;
                const int ths = ceil_div(th, subs);
                if ((subs - 1) * ths >= th) continue;                      // an empty last sub-tile
                const int thi = (ths - 1) * stride + 2 * dil + 1;
                const int twi = (tw - 1) * stride + 2 * dil + 1;
                if (thi > 256 || twi > 256) continue;
                const long long box = (long long)thi * twi * g.cbox * 2;
                const long long stage = ((box + 127) & ~127ll) + wgt_stage;
                // segments: 4-pixel (8 when half) column strips x seg_rows rows.  They are handed out dynamically across
                // the items in flight (A stages x segments >= 16 keeps the 10 warps busy); ~4-5 rows amortise the window preload
                const int spr = ceil_div(tw, sw);
                // (dilated blocks: a segment walks one residue class of rows, ths / dil rows per class)
                const int rstep = stride == 1 ? dil : 1;
                const int class_rows = ceil_div(ths, rstep);
                int pieces = ceil_div(class_rows, 5);                                // row chunks per class
                if (pieces * spr * subs * rstep < 8) pieces = ceil_div(8, spr * subs * rstep);   // >= 16 segments in flight with 2 A stages
                if (pieces > class_rows) pieces = class_rows;
                const int seg_rows = ceil_div(class_rows, pieces);
                int segs = 0;
                for (int c = 0; c < rstep && c < ths; ++c) segs += spr * ceil_div(ceil_div(ths - c, rstep), seg_rows);
                if (segs > 64 || seg_rows > 255 || tw > 255 || ths > 255) continue;
                const long long room = SEP_SMEM_MAX - fixed;
                const int pst = (int)(room / stage);
                if (pst < 2 || pst < subs + 1) continue;
                const long long tiles = (long long)ceil_div(g.ho, th) * ceil_div(g.wo, tw);
                // per k-block cycles.  A depthwise step (one strip row, one warp) issues ~45 + 10 per window column
                // instructions (+ ~1.3 per preloaded element and ~120 per segment hand-out); all warps together set the issue
                // time (4 schedulers, 25 % imbalance), half a segment's latency (~1.6 cycles per instruction) is exposed.
                // Tensor pipe: 2 cycles per output column.  Patch fill at ~40 B/clk.
                const double step = 45.0 + 10.0 * ncols * (slide ? (stride + 2.0) / 3.0 : 1.0), prol = 1.3 * pre * ncols + 120.0;
                const double lat = 0.5 * (seg_rows * step + prol) * 1.6;
                const double issue = 1.25 * (double)subs * (spr * ths * step + segs * prol) / 4.0;
                const double dwc = lat > issue ? lat : issue;
                const double mma = 2.0 * g.n_tile;                          // per k-block, all column blocks
                const double fill = (double)subs * stage / 40.0;
                double per_kb = dwc > mma ? dwc : mma;
                if (fill > per_kb) per_kb = fill;
                per_kb += 0.25 * fill;                                     // halo re-reads load the L2 -> SM path
                if (pst < 3 * subs) per_kb *= 1.08;                        // shallow prefetch (measured: two stages of a compact tile beat three of a thin one)
                // per tile: pipeline hand-off + an epilogue whose work is 128 rows x n_tile whatever the tile covers
                const double cost = (double)tiles * (g.kblocks * per_kb + 400.0 + 200.0 * g.panels);
                if (cost < best) {
                    best = cost;
                    g.th = th; g.tw = tw; g.subs = subs; g.ths = ths; g.thi = thi; g.twi = twi; g.spr = spr; g.seg_rows = seg_rows;
                    g.segs_per_sub = segs;
                    g.patch_box_bytes = (unsigned)box;
                    g.wgt_off = (unsigned)((box + 127) & ~127ll);
                    g.patch_stage_bytes = (unsigned)stage;
                }
            }
        }
    }
    PN_CHECK_ARG(best < 1e300, "pn_sepconv_block: no tile shape fits (cin %d stride %d dilation %d)", k, stride, dil);
    {   // segment table: strips x residue classes x row chunks
        const int rstep = stride == 1 ? dil : 1;
        int nseg = 0;
        for (int c = 0; c < rstep && c < g.ths; ++c) {
            const int rows_c = ceil_div(g.ths - c, rstep);
            for (int r = 0; r < rows_c; r += g.seg_rows)
                for (int cs = 0; cs < g.spr; ++cs) {
                    const int nrow = rows_c - r < g.seg_rows ? rows_c - r : g.seg_rows;
                    g.segtab[nseg++] = (unsigned)(cs * sw) | (unsigned)(c + r * rstep) << 8 | (unsigned)nrow << 16;
                }
        }
        PN_CHECK_ARG(nseg == g.segs_per_sub, "pn_sepconv_block: internal segment accounting error (%d vs %d)", nseg, g.segs_per_sub);
    }
    g.tiles_x = ceil_div(g.wo, g.tw);
    g.tiles_y = ceil_div(g.ho, g.th);
    g.tiles = (long long)n * g.tiles_x * g.tiles_y * g.n_tiles;
    // ---- shared-memory carve-up: W ring, A ring, output staging panels, patch ring, bias, barriers
    const long long bias_bytes = ((long long)g.n_tiles * g.panels * 64 * 4 + 127) & ~127ll;
    const long long avail = SEP_SMEM_MAX - 1024 - 640 - bias_bytes - dww_bytes;   // alignment slack, barrier block (SepBars::total)
    auto fits = [&](int pst, int wst, int ast, int stg) {
        return (long long)wst * g.w_stage_bytes + (long long)ast * SEP_A_BYTES + (long long)stg * SEP_STG_BYTES +
                   (long long)pst * g.patch_stage_bytes <= avail;
    };
    int bestp = -1;
    // Direct epilogue (stg = 0): stores straight from registers, no staging panels, no CTA barriers, TMEM loads pipelined; the
    // 16-32 KB of the panels go to the rings.  It is the default for single-accumulator tiles (n_tile > 256: the epilogue
    // cannot overlap the next tile's MMAs there, so its barrier hand-offs are pure stall) -- measured on B200, fused block
    // alone: 256 -> 512 stride 2 at 65x65 95 -> 72 us, 192 -> 384 stride 2 at 33x33 110 -> 94 us, 384 -> 384 at 17x17 128 -> 113 us,
    // 512 -> 512 at 33x33 68 -> 65 us.  Double-buffered tiles keep the staged TMA-store epilogue (it overlaps the main loop;
    // direct stores are scattered 32-byte pieces and measured 10 % slower there).
    const bool direct = g.acc_bufs == 1;
    const int max_a1 = direct ? 4 : 3;
    for (int stg = direct ? 0 : 2; stg >= (direct ? 0 : 1); --stg)
        for (int ast = max_a1; ast >= 2; --ast) {
            for (int wst = g.w_res ? min_w : SEP_MAX_W; wst >= min_w; --wst)
                for (int pst = SEP_MAX_P; pst >= 2 && pst >= g.subs + 1; --pst) {
                    if (!fits(pst, wst, ast, stg)) continue;
                    const int want = 3 * g.subs > SEP_MAX_P ? SEP_MAX_P : 3 * g.subs;
                    // deep patch prefetch first, then one spare W block, a third A stage, a second staging panel
                    // (direct epilogue: a fourth A stage lets the depthwise warps run further ahead while the accumulator drains;
                    // it measured better than a fourth W block)
                    const int score = (pst >= want ? 1000 : pst * 100) + (wst > min_w + (direct ? 0 : 1) ? min_w + (direct ? 0 : 1) : wst) * 20 +
                                      ast * (direct ? 24 : 8) + stg * 4 + (pst > want ? 1 : 0);
                    if (score > bestp) {
                        bestp = score;
                        g.p_stages = pst; g.w_stages = wst; g.a_stages = ast; g.stg_bufs = stg;
                    }
                }
        }
    PN_CHECK_ARG(bestp >= 0, "pn_sepconv_block: shared memory budget exceeded");
    // 512-column tiles have a single accumulator: the epilogue cannot overlap the next tile's MMAs, so what pays is a
    // short epilogue (two staging panels keep the TMA stores in flight) and a third A stage for the depthwise warps to
    // run ahead into -- worth more than a third patch stage (measured: 84 -> 77 us on the 512 -> 512 blocks)
    if (!direct && g.n_halves == 2 && g.subs == 1 && fits(2, min_w, 3, 2)) { g.p_stages = 2; g.w_stages = min_w; g.a_stages = 3; g.stg_bufs = 2; }
    {   // ring depths: the table's (p = 0: the rule above), or forced with PN_SEP_STAGES="p,w,a,stg"
        int fp = 0, fw = 0, fa = 0, fs = 0;
        bool have = false;
        if (tuned && tuned->p > 0 && g.th == tuned->th && g.tw == tuned->tw && g.subs == tuned->subs) { fp = tuned->p; fw = tuned->w; fa = tuned->a; fs = tuned->stg; have = true; }
        if (const char *force = getenv("PN_SEP_STAGES")) have = sscanf(force, "%d,%d,%d,%d", &fp, &fw, &fa, &fs) == 4;
        if (have && fp >= g.subs + 1 && fp <= SEP_MAX_P && fw >= 1 &&
            fw <= SEP_MAX_W && fa >= 2 && fa <= SEP_MAX_A && fs >= 0 && fs <= 2 && fits(fp, fw, fa, fs)) {
            g.p_stages = fp; g.w_stages = fw; g.a_stages = fa; g.stg_bufs = fs;
        }
    }
    if (g.w_res && g.w_stages != g.kblocks * g.n_halves) g.w_res = 0;   // (a forced ring depth: back to the ring)
    // Depthwise warp teams (see the kernel): two items in flight need a patch stage per team and sub-tile plus one ahead, an A
    // stage per team plus the one the MMAs read, and -- for the parity of a barrier a team returns to -- a patch ring at least as
    // deep as the A ring (an item whose A stage is free has had the patch stage's previous user consumed).  PN_SEP_TEAMS=1 / 2.
    g.teams = (SEP_DW_WARPS % 2 == 0 && g.p_stages >= 2 * g.subs + 1 && g.a_stages >= 3 && g.p_stages >= g.a_stages) ? 2 : 1;
    {
        const char *e = getenv("PN_SEP_TEAMS");
        const int v = e ? atoi(e) : (tuned && tuned->p > 0 && g.th == tuned->th && g.tw == tuned->tw && g.subs == tuned->subs) ? tuned->teams : 0;
        if (v == 1 || (v == 2 && SEP_DW_WARPS % 2 == 0 && g.p_stages >= 2 * g.subs && g.a_stages >= 2 && g.p_stages >= g.a_stages)) g.teams = v;
    }
    static_assert(SepBars::total <= 640, "barrier block exceeds its reserve");
    g.off_a = (unsigned)g.w_stages * g.w_stage_bytes;
    g.off_stg = g.off_a + (unsigned)g.a_stages * SEP_A_BYTES;
    g.off_patch = g.off_stg + (unsigned)g.stg_bufs * SEP_STG_BYTES;
    g.off_bias = g.off_patch + (unsigned)g.p_stages * g.patch_stage_bytes;
    g.off_dww = g.off_bias + (unsigned)bias_bytes;
    g.off_bar = g.off_dww + (unsigned)dww_bytes;
    op->smem_bytes = (int)(g.off_bar + SepBars::total + 1024);
    PN_CHECK_ARG(op->smem_bytes <= SEP_SMEM_MAX, "pn_sepconv_block: internal smem accounting error (%d)", op->smem_bytes);
    static_assert(sizeof(SepGeom) <= sizeof(op->geom), "SepOp::geom too small");
    memcpy(op->geom, &g, sizeof(g));
    op->cb = cb; op->stride = stride; op->dil = dil;
    op->ho = g.ho; op->wo = g.wo;
    op->n = n; op->h = h; op->w = wd; op->k = k; op->nc = nc;
    return PN_OK;
}

int sep_prepare(SepOp *op, const void *x, const float *dw_w, const float *dw_b, const void *pw_w, void *y, int n, int h,
                int wd, int k, int nc, int stride, int dil) {
    PN_CHECK_ARG(x && dw_w && dw_b && pw_w && y, "pn_sepconv_block: null pointer");
    PN_CHECK_ARG(((uintptr_t)x & 15) == 0 && ((uintptr_t)y & 15) == 0 && ((uintptr_t)pw_w & 15) == 0 && ((uintptr_t)dw_w & 15) == 0 &&
                     ((uintptr_t)dw_b & 15) == 0,
                 "pn_sepconv_block: pointers must be 16-byte aligned");
    int rc = sep_geometry(op, n, h, wd, k, nc, stride, dil);
    if (rc != PN_OK) return rc;
    if (op->warp_kind) {
        op->dw_w = dw_w; op->dw_b = dw_b; op->pw_w = pw_w; op->y = y;
        return sepwarp_prepare(&op->warp, x, n, h, wd, k, nc, stride);
    }
    if (op->tc_kind) {
        op->dw_w = dw_w; op->dw_b = dw_b; op->pw_w = pw_w; op->y = y;
        return septc_prepare(&op->tc, x, pw_w, n, h, wd, k, nc, dil);
    }
    op->y = y;                                                       // the direct-store epilogue writes through the plain pointer
    op->dw_w = dw_w; op->dw_b = dw_b;                                // (resident depthwise weights are read through plain pointers too)
    SepGeom g;
    memcpy(&g, op->geom, sizeof(g));
    {   // input patches: (C, W, H, N) bf16, box [cb, twi, thi, 1], no swizzle, OOB -> 0
        const uint64_t dims[4] = {(uint64_t)k, (uint64_t)wd, (uint64_t)h, (uint64_t)n};
        const uint64_t strides[3] = {(uint64_t)k * 2, (uint64_t)wd * k * 2, (uint64_t)h * wd * k * 2};
        const uint32_t box[4] = {(uint32_t)g.cbox, (uint32_t)g.twi, (uint32_t)g.thi, 1u};
        if ((rc = encode_tmap(op->tmap_x, x, 2, 4, dims, strides, box, 0)) != PN_OK) return rc;
    }
    {   // depthwise weights [9, K] fp32, box [64, 9]; bias [1, K] fp32, box [64, 1]
        const uint64_t dims[2] = {(uint64_t)k, 9};
        const uint64_t strides[1] = {(uint64_t)k * 4};
        const uint32_t box[2] = {64u, 9u};
        if ((rc = encode_tmap(op->tmap_dww, dw_w, 4, 2, dims, strides, box, 0)) != PN_OK) return rc;
        const uint64_t bdims[2] = {(uint64_t)k, 1};
        const uint32_t bbox[2] = {64u, 1u};
        if ((rc = encode_tmap(op->tmap_dwb, dw_b, 4, 2, bdims, strides, bbox, 0)) != PN_OK) return rc;
    }
    {   // pointwise weights [Nc, K] bf16, box [64, n_tile], 128B swizzle
        const uint64_t dims[2] = {(uint64_t)k, (uint64_t)nc};
        const uint64_t strides[1] = {(uint64_t)k * 2};
        const uint32_t box[2] = {64u, (uint32_t)g.n_half};
        if ((rc = encode_tmap(op->tmap_w, pw_w, 2, 2, dims, strides, box, 3)) != PN_OK) return rc;
    }
    {   // output (C, W, H, N) bf16, box [64, tw, th, 1], 128B swizzle
        const uint64_t dims[4] = {(uint64_t)nc, (uint64_t)g.wo, (uint64_t)g.ho, (uint64_t)n};
        const uint64_t strides[3] = {(uint64_t)nc * 2, (uint64_t)g.wo * nc * 2, (uint64_t)g.ho * g.wo * nc * 2};
        const uint32_t box[4] = {64u, (uint32_t)g.tw, (uint32_t)g.th, 1u};
        if ((rc = encode_tmap(op->tmap_y, y, 2, 4, dims, strides, box, 3)) != PN_OK) return rc;
    }
    return PN_OK;
}

template <int S, int D, bool HALF>
static int sep_launch_t(const SepOp *op, const SepGeom &g, const float *pw_bias, cudaStream_t st) {
    static DeviceOnce once;                                       // per device: attribute set
    const int dev = current_device();
    auto kern = sepconv_kernel<S, D, HALF>;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;   // PDL (common.cuh: launch_pdl)
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.blockDim = dim3(SEP_THREADS, 1, 1);
    cfg.dynamicSmemBytes = (size_t)op->smem_bytes;
    cfg.stream = st;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    if (!once.get(dev)) {
        PN_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SEP_SMEM_MAX));
        once.set(dev, 1);
    }
    const long long units = num_sms();                            // persistent: one CTA per SM
    cfg.gridDim = dim3((unsigned)(g.tiles < units ? g.tiles : units), 1, 1);
    PN_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kern, *reinterpret_cast<const CUtensorMap *>(op->tmap_x),
                                     *reinterpret_cast<const CUtensorMap *>(op->tmap_dww), *reinterpret_cast<const CUtensorMap *>(op->tmap_dwb),
                                     *reinterpret_cast<const CUtensorMap *>(op->tmap_w), *reinterpret_cast<const CUtensorMap *>(op->tmap_y),
                                     pw_bias, reinterpret_cast<__nv_bfloat16 *>(op->y), op->dw_w, op->dw_b, g));
    return PN_OK;
}

int sep_launch(const SepOp *op, const float *pw_bias, cudaStream_t st) {
    PN_CHECK_ARG(op && pw_bias, "pn_sepconv_block: null pointer");
    if (op->warp_kind) return sepwarp_launch(&op->warp, op->dw_w, op->dw_b, op->pw_w, pw_bias, op->y, st);
    if (op->tc_kind) return septc_launch(&op->tc, op->dw_w, op->dw_b, pw_bias, op->y, st);
    SepGeom g;
    memcpy(&g, op->geom, sizeof(g));
    if (op->stride == 2) return sep_launch_t<2, 1, false>(op, g, pw_bias, st);
    if (g.half) return sep_launch_t<1, 1, true>(op, g, pw_bias, st);
    if (op->dil == 1) return sep_launch_t<1, 1, false>(op, g, pw_bias, st);
    if (op->dil == 2) return sep_launch_t<1, 2, false>(op, g, pw_bias, st);
    return sep_launch_t<1, 4, false>(op, g, pw_bias, st);
}

void sep_describe(const SepOp *op, char *out, size_t cap) {
    if (op->tc_kind) {
        septc_describe(&op->tc, out, cap);
        return;
    }
    if (op->warp_kind) {
        SepWarpOp w;
        if (sepwarp_geometry(&w, op->n, op->h, op->w, op->k, op->nc, op->stride) == PN_OK) sepwarp_describe(&w, out, cap);
        else snprintf(out, cap, "warp-autonomous (geometry unavailable)");
        return;
    }
    SepGeom g;
    memcpy(&g, op->geom, sizeof(g));
    snprintf(out, cap, "%stile %dx%d subs %d box %dx%d segs %d x %d rows n_tile %d(%dx%d) x%d kblocks %d teams %d stages p%d w%d%s a%d stg%d smem %d tiles %lld",
             g.half ? "half " : "", g.th, g.tw, g.subs, g.thi, g.twi, g.segs_per_sub, g.seg_rows, g.n_tile, g.n_halves, g.n_half, g.n_tiles, g.kblocks, g.teams, g.p_stages,
             g.w_stages, g.w_res ? "r" : "", g.a_stages, g.stg_bufs, op->smem_bytes, g.tiles);
}

}  // namespace pn

#ifdef PN_SEP_TRACE
// debug only: trace buffer = 4 roles x cap events x 4 stamps (int64), zero-filled by the caller
extern "C" int pn_debug_sep_trace(long long *buf, int cap) {
    if (cudaMemcpyToSymbol(pn::g_sep_trace, &buf, sizeof(buf)) != cudaSuccess) return -2;
    if (cudaMemcpyToSymbol(pn::g_sep_trace_cap, &cap, sizeof(cap)) != cudaSuccess) return -2;
    return 0;
}
#endif
