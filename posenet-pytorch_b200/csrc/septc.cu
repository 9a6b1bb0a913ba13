// B3 + B4 fused with the DEPTHWISE ON THE TENSOR PIPE -- one SeperableConv block (posenet/models/mobilenet_v1.py:57-68 of the
// reference), stride 1, dilation 1 / 2, cin = cout = 256:
//     y = relu6( pointwise1x1( relu6( depthwise3x3(x; dilation) + b_dw ) ) + b_pw )
// The CUDA-core depthwise of sepconv.cu is issue-bound (~12 thread-instructions per output).  Here the 3x3 depthwise is nine
// tcgen05.mma per 16-channel group against block-diagonal weight tiles:
//     D[128 positions, 16 ch] += A_tap[128 positions, 16 ch] * diag(w_tap[16 ch])            (M = 128, N = 16, K = 16)
// where A_tap is a SHIFTED VIEW of the TMA-written input patch: the patch is a flat array of pixels (one 128-byte swizzled row
// per pixel and 64-channel k-block) with row pitch `wp`, so the tap (dy, dx) of 128 consecutive flat positions is the same
// array advanced by (dy * wp + dx) * dilation rows -- a descriptor start-address change, no data movement (the UMMA swizzle is a
// function of the absolute shared-memory address, verified by csrc/dwtc_probe.cu).  Positions whose column falls into the
// halo part of the pitch are computed and dropped.  The depthwise accumulator (TMEM, fp32) is read back once per k-block by
// four converter warps (+ bias, ReLU6 -> bf16) and stored back into TMEM as the A operand of the pointwise MMA
// (tcgen05.mma with A in tensor memory), so the intermediate never touches shared memory or HBM.
// What bounds it: every tap MMA re-reads its 4 KB A slice from shared memory (9 x the patch per k-block, ~1150 cycles per
// 128 positions x 64 channels at 128 B/clk) -- about the CUDA-core kernel's issue time, but the SM's issue slots stay free.
//
// Work unit: 128 consecutive flat positions ("chunk") of one column band of one image.  Two step sequences per CTA:
//   depthwise step d = (unit, k-block)            patch stage d % PS, diag / depthwise-accumulator buffer d % 2
//   pointwise step s = (unit, k-block)            W stage s % WS, A operand s % 4
// A operands (32 TMEM columns each): 4 buffers used round-robin, so the depthwise runs up to four k-blocks ahead of the
// pointwise MMAs (covers the epilogue of the single-buffered accumulator).
//   warp 0        patch producer  TMA box [64 ch, wp, rows_box] (OOB zero fill == zero padding), 128B swizzle
//   warp 15       W producer      pointwise weight tile [256 x 64] (128B swizzle)
//   warps 16-17   depthwise MMA   warp 16 + w issues the 2 x 9 tap MMAs of channel groups 2w, 2w+1; commits release patch / diag stages
//   warps 2-5     converters      tcgen05.ld depthwise accumulator -> bias, ReLU6, bf16x2 -> tcgen05.st (A operand)
//   warp 1        pointwise MMA   4 MMAs per step, A from TMEM; commits release the W stage, the A operand, and signal the epilogue
//   warps 6-13    epilogue        tcgen05.ld 32 accumulator columns -> bias, ReLU6 -> bf16 -> warp-private staging -> coalesced
//                                 predicated 16-byte global stores
//   warp 14       diag writer     the 9 x 4 diagonal weight tiles of the next k-block (576 bf16 values into pre-zeroed tiles)
// TMEM (512 columns): accumulator at 0, A operands 4 x 32 at 256, depthwise accumulators 2 x 64 at 384.
#include <cuda.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "ptx.cuh"

namespace pn {

constexpr int TCS_WARPS = 18;
constexpr int TCS_THREADS = TCS_WARPS * 32;
constexpr int TCS_MAX_P = 4, TCS_MAX_W = 4, TCS_A_BUFS = 4;
constexpr int TCS_DIAG_BYTES = 9 * 16 * 128;          // nine [16 x 64] bf16 tiles
constexpr int TCS_STG_BYTES = 32 * 64;                // per epilogue warp: 32 rows x 32 bf16
constexpr int TCS_EPI_WARPS = 8;
constexpr int TCS_DW_ISSUERS = 2;
constexpr int TCS_SMEM_MAX = 232448;
constexpr uint32_t TCS_A_COL = 256, TCS_DW_COL = 384;
// Every mbarrier poll is a shared-memory wavefront, and the shared-memory pipe is what bounds this kernel (tensor-operand
// fetches): waiting warps sleep between polls (ns) instead of re-polling every few tens of cycles.
constexpr unsigned TCS_SLEEP_PRODUCER = 100, TCS_SLEEP_MMA = 32, TCS_SLEEP_CONVERT = 64, TCS_SLEEP_EPI = 300, TCS_SLEEP_DIAG = 200;

struct TcsGeom {
    int k, nc, h, w, n_img, dil;
    int wp, tw, bands, rows_box, chunks;
    int kblocks;
    int p_stages, w_stages;
    unsigned patch_bytes, patch_stage_bytes, w_stage_bytes;
    unsigned off_diag, off_patch, off_stg, off_dww, off_dwb, off_pwb, off_bar;
    unsigned magic_wp;
    long long units;
};

struct TcsBars {
    static constexpr int patch_full = 0, patch_empty = 32, w_full = 64, w_empty = 96, diag_full = 128, diag_empty = 144,
                         dw_full = 160, dw_free = 176, a_full = 192, a_empty = 256, tfull = 320, tempty = 336, tmem_slot = 352,
                         total = 368;
};

__device__ __forceinline__ uint64_t tcs_desc(uint32_t saddr) {          // K-major SWIZZLE_128B, 8-row groups 1024 B apart
    return (uint64_t)((saddr & 0x3FFFF) >> 4) | (1ull << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
__device__ __forceinline__ uint32_t tcs_idesc(int n) {                   // D f32, A/B bf16, K-major, M = 128
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}
__device__ __forceinline__ void tcs_mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
        "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tcs_st32(uint32_t taddr, const uint32_t *v) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
        "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]),
        "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]),
        "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]),
        "r"(v[31])
        : "memory");
}
__device__ __forceinline__ void tcs_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ float4 tcs_lds_f4(uint32_t addr) {
    float4 r;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "r"(addr));
    return r;
}
__device__ __forceinline__ uint32_t tcs_lds_u16(uint32_t addr) {
    unsigned short r;
    asm volatile("ld.shared.u16 %0, [%1];" : "=h"(r) : "r"(addr));
    return r;
}
__device__ __forceinline__ void tcs_sts_u16(uint32_t addr, uint32_t v) {
    asm volatile("st.shared.u16 [%0], %1;" ::"r"(addr), "h"((unsigned short)v) : "memory");
}
__device__ __forceinline__ void tcs_stg_v4(void *p, const uint4 &v) {
    asm volatile("st.global.v4.b32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// Timeline trace (diagnostics build only: -DPN_TCS_TRACE, tools/trace_septc.py): CTA 0 stamps clock64 at the hand-offs of its
// first `cap` steps into [role][step][4] once a buffer has been registered with pn_debug_tcs_trace.
#ifdef PN_TCS_TRACE
__device__ long long *g_tcs_trace = nullptr;
__device__ int g_tcs_trace_cap = 0;
#define TCS_TR(role, step, ev)                                                                         \
    do {                                                                                                \
        if (tr && (step) < tr_cap) tr[(((long long)(role)) * tr_cap + (step)) * 4 + (ev)] = clock64();  \
    } while (0)
#else
#define TCS_TR(role, step, ev) do { } while (0)
#endif

__global__ void __launch_bounds__(TCS_THREADS, 1)
septc_kernel(const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_w, const float *__restrict__ dw_w,
             const float *__restrict__ dw_b, const float *__restrict__ pw_b, __nv_bfloat16 *__restrict__ y, const TcsGeom g) {
    extern __shared__ uint8_t tcs_smem_raw[];
    const uint32_t base = (smem_u32(tcs_smem_raw) + 1023u) & ~1023u;
    uint8_t *gen = tcs_smem_raw + (base - smem_u32(tcs_smem_raw));
    const uint32_t bars = base + g.off_bar;
    auto bar = [&](int which, int s) { return bars + (uint32_t)which + 8u * (uint32_t)s; };
    auto w_addr = [&](int s) { return base + (uint32_t)s * g.w_stage_bytes; };
    auto p_addr = [&](int s) { return base + g.off_patch + (uint32_t)s * g.patch_stage_bytes; };
    auto d_addr = [&](int s) { return base + g.off_diag + (uint32_t)s * TCS_DIAG_BYTES; };
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long ustride = gridDim.x;
    const int my_units = (long long)blockIdx.x < g.units ? (int)((g.units - blockIdx.x + ustride - 1) / ustride) : 0;
    const int per_img = g.bands * g.chunks;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmap_x);
        tma_prefetch_desc(&tmap_w);
        for (int s = 0; s < TCS_MAX_P; ++s) {
            mbar_init(bar(TcsBars::patch_full, s), 1);
            mbar_init(bar(TcsBars::patch_empty, s), TCS_DW_ISSUERS);      // one tcgen05.commit per depthwise issuer
            mbar_init(bar(TcsBars::w_full, s), 1);
            mbar_init(bar(TcsBars::w_empty, s), 1);
        }
        for (int s = 0; s < 2; ++s) {
            mbar_init(bar(TcsBars::diag_full, s), 1);
            mbar_init(bar(TcsBars::diag_empty, s), TCS_DW_ISSUERS);
            mbar_init(bar(TcsBars::dw_full, s), TCS_DW_ISSUERS);
            mbar_init(bar(TcsBars::dw_free, s), 128);
            mbar_init(bar(TcsBars::tfull, s), 1);
            mbar_init(bar(TcsBars::tempty, s), TCS_EPI_WARPS * 32);
        }
        for (int s = 0; s < TCS_A_BUFS; ++s) {
            mbar_init(bar(TcsBars::a_full, s), 128);
            mbar_init(bar(TcsBars::a_empty, s), 1);
        }
        mbar_fence_init();
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(bars + (uint32_t)TcsBars::tmem_slot) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    // weights are not produced by the previous layer: stage them before griddepcontrol.wait
    for (uint32_t o = threadIdx.x * 16; o < 2u * TCS_DIAG_BYTES; o += TCS_THREADS * 16) st_shared_v4(base + g.off_diag + o, 0, 0, 0, 0);
    {
        unsigned short *sdww = reinterpret_cast<unsigned short *>(gen + g.off_dww);
        for (int i = threadIdx.x; i < 9 * g.k; i += TCS_THREADS) {
            const __nv_bfloat16 b = __float2bfloat16_rn(__ldg(dw_w + i));
            sdww[i] = *reinterpret_cast<const unsigned short *>(&b);
        }
        float *sdwb = reinterpret_cast<float *>(gen + g.off_dwb);
        for (int i = threadIdx.x; i < g.k; i += TCS_THREADS) sdwb[i] = __ldg(dw_b + i);
        float *spwb = reinterpret_cast<float *>(gen + g.off_pwb);
        for (int i = threadIdx.x; i < g.nc; i += TCS_THREADS) spwb[i] = __ldg(pw_b + i);
    }
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    pdl_launch_dependents();                                  // after the TMEM allocation is made (see stem.cu): a dependent CTA must not allocate first
    pdl_wait();
    const uint32_t tmem = *reinterpret_cast<volatile uint32_t *>(gen + g.off_bar + TcsBars::tmem_slot);
#ifdef PN_TCS_TRACE
    long long *tr = blockIdx.x == 0 ? g_tcs_trace : nullptr;
    const int tr_cap = g_tcs_trace_cap;
#endif
    if (warp == 0) {
        // ===================== patch producer =====================
        if (lane == 0) {
            int ps = 0, d = 0;
            uint32_t pph = 0;
            for (long long u = blockIdx.x; u < g.units; u += ustride) {
                const int img = (int)(u / per_img), rem = (int)(u - (long long)img * per_img);
                const int band = rem / g.chunks, chunk = rem - band * g.chunks;
                const int row0 = (int)__umulhi((uint32_t)(chunk * 128), g.magic_wp);
                const int x_org = band * g.tw - g.dil, y_org = row0 - g.dil;
                for (int kb = 0; kb < g.kblocks; ++kb, ++d) {
                    mbar_wait_backoff(bar(TcsBars::patch_empty, ps), pph ^ 1u, TCS_SLEEP_PRODUCER);
                    TCS_TR(0, d, 0);
                    mbar_expect_tx(bar(TcsBars::patch_full, ps), g.patch_bytes);
                    tma_load_4d(p_addr(ps), &tmap_x, bar(TcsBars::patch_full, ps), kb * 64, x_org, y_org, img);
                    if (++ps == g.p_stages) { ps = 0; pph ^= 1u; }
                }
            }
        }
    } else if (warp == 15) {
        // ===================== W producer =====================
        if (lane == 0) {
            int ws = 0, s = 0;
            uint32_t wph = 0;
            for (int i = 0; i < my_units; ++i)
                for (int kb = 0; kb < g.kblocks; ++kb, ++s) {
                    mbar_wait_backoff(bar(TcsBars::w_empty, ws), wph ^ 1u, TCS_SLEEP_PRODUCER);
                    TCS_TR(0, s, 1);
                    mbar_expect_tx(bar(TcsBars::w_full, ws), g.w_stage_bytes);
                    tma_load_2d(w_addr(ws), &tmap_w, bar(TcsBars::w_full, ws), kb * 64, 0);
                    if (++ws == g.w_stages) { ws = 0; wph ^= 1u; }
                }
        }
    } else if (warp == 1) {
        // ===================== pointwise MMA issuer (A operand in TMEM) =====================
        if (lane == 0) {
            const uint32_t idesc_n = tcs_idesc(g.nc);
            const uint64_t desc_hi = tcs_desc(0);
            int pws = 0, s = 0;
            uint32_t pwph = 0;
            for (int i = 0; i < my_units; ++i)
                for (int kb = 0; kb < g.kblocks; ++kb, ++s) {
                    const int ai = s & (TCS_A_BUFS - 1);
                    const uint32_t use = (uint32_t)s / TCS_A_BUFS;            // earlier uses of A operand ai
                    TCS_TR(1, s, 0);
                    if (kb == 0) mbar_wait_backoff(bar(TcsBars::tempty, 0), ((uint32_t)i & 1u) ^ 1u, TCS_SLEEP_MMA);
                    mbar_wait_backoff(bar(TcsBars::w_full, pws), pwph, TCS_SLEEP_MMA);
                    TCS_TR(1, s, 1);
                    mbar_wait_backoff(bar(TcsBars::a_full, ai), use & 1u, TCS_SLEEP_MMA);
                    TCS_TR(1, s, 2);
                    tc_fence_after();
                    const uint32_t w0 = (w_addr(pws) & 0x3FFFF) >> 4;
                    const uint32_t acol = tmem + TCS_A_COL + (uint32_t)(ai * 32);
#pragma unroll
                    for (int k4 = 0; k4 < 4; ++k4)
                        tcs_mma_ts(tmem, acol + k4 * 8, desc_hi | (uint64_t)(w0 + k4 * 2), idesc_n, (kb > 0 || k4 > 0));
                    tc_commit(bar(TcsBars::w_empty, pws));
                    tc_commit(bar(TcsBars::a_empty, ai));
                    if (kb == g.kblocks - 1) tc_commit(bar(TcsBars::tfull, 0));
                    TCS_TR(1, s, 3);
                    if (++pws == g.w_stages) { pws = 0; pwph ^= 1u; }
                }
        }
    } else if (warp >= 16) {
        // ===================== depthwise MMA issuers: warp 16 + w owns the 16-channel groups 2w and 2w + 1 =====================
        if (lane == 0) {
            const int w2 = warp - 16;
            const uint32_t idesc16 = tcs_idesc(16);
            uint32_t tap[9];                                     // tap shifts in 16-byte descriptor units
#pragma unroll
            for (int t = 0; t < 9; ++t) tap[t] = (uint32_t)((t / 3) * g.dil * g.wp + (t % 3) * g.dil) * 8u + (uint32_t)w2 * 4u;
            const uint64_t desc_hi = tcs_desc(0);
            int dps = 0, d = 0;
            uint32_t dpph = 0;
            for (long long u = blockIdx.x; u < g.units; u += ustride) {
                const int chunk = (int)(u % per_img) % g.chunks;
                const int row0 = (int)__umulhi((uint32_t)(chunk * 128), g.magic_wp);
                const uint32_t qoff = (uint32_t)(chunk * 128 - row0 * g.wp) * 8u;
                for (int kb = 0; kb < g.kblocks; ++kb, ++d) {
                    const int db = d & 1;
                    const uint32_t dph = (uint32_t)(d >> 1) & 1u;
                    mbar_wait_backoff(bar(TcsBars::dw_free, db), dph ^ 1u, TCS_SLEEP_MMA);            // the converters have read accumulator db (step d - 2)
                    if (w2 == 0) TCS_TR(2, d, 0);
                    mbar_wait_backoff(bar(TcsBars::patch_full, dps), dpph, TCS_SLEEP_MMA);
                    if (w2 == 0) TCS_TR(2, d, 1);
                    mbar_wait_backoff(bar(TcsBars::diag_full, db), dph, TCS_SLEEP_MMA);
                    if (w2 == 0) TCS_TR(2, d, 2);
                    tc_fence_after();
                    const uint32_t a0 = ((p_addr(dps) & 0x3FFFF) >> 4) + qoff, b0 = ((d_addr(db) & 0x3FFFF) >> 4) + (uint32_t)w2 * 4u;
                    const uint32_t dcol = tmem + TCS_DW_COL + (uint32_t)db * 64u + (uint32_t)w2 * 32u;
#pragma unroll
                    for (int gq = 0; gq < 2; ++gq)
#pragma unroll
                        for (int t = 0; t < 9; ++t)
                            tc_mma_bf16(dcol + gq * 16, desc_hi | (uint64_t)(a0 + tap[t] + gq * 2), desc_hi | (uint64_t)(b0 + t * 128 + gq * 2),
                                        idesc16, t > 0);
                    tc_commit(bar(TcsBars::patch_empty, dps));
                    tc_commit(bar(TcsBars::diag_empty, db));
                    tc_commit(bar(TcsBars::dw_full, db));
                    if (w2 == 0) TCS_TR(2, d, 3);
                    if (++dps == g.p_stages) { dps = 0; dpph ^= 1u; }
                }
            }
        }
    } else if (warp < 6) {
        // ===================== converters: depthwise accumulator -> A operand =====================
        const uint32_t lane_off = (uint32_t)((warp & 3) * 32) << 16;
        const uint32_t sdwb = base + g.off_dwb;
        int d = 0;
        for (int i = 0; i < my_units; ++i)
            for (int kb = 0; kb < g.kblocks; ++kb, ++d) {
                const int b = d & 1;
                const int a = i * g.kblocks + kb, ai = a & (TCS_A_BUFS - 1);   // A operand of step d (== d, but written from (i, kb):
                const uint32_t use = (uint32_t)a / TCS_A_BUFS;                 // with the counter itself ptxas spills in this kernel)
                mbar_wait_backoff(bar(TcsBars::dw_full, b), (uint32_t)(d >> 1) & 1u, TCS_SLEEP_CONVERT);
                if (threadIdx.x == 64) TCS_TR(3, d, 0);
                tc_fence_after();
                uint32_t v[32], pk[32];
#pragma unroll
                for (int hf = 0; hf < 2; ++hf) {
                    tc_ld32(tmem + lane_off + TCS_DW_COL + (uint32_t)(b * 64 + hf * 32), v);
                    tc_ld_wait();
                    if (hf == 1) {                                  // accumulator b may be overwritten by depthwise step d + 2
                        tc_fence_before();
                        mbar_arrive(bar(TcsBars::dw_free, b));
                    }
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const float4 bb = tcs_lds_f4(sdwb + (uint32_t)(kb * 64 + hf * 32 + j * 4) * 4u);
                        pk[hf * 16 + 2 * j] = relu6_bf16x2(__uint_as_float(v[4 * j]) + bb.x, __uint_as_float(v[4 * j + 1]) + bb.y);
                        pk[hf * 16 + 2 * j + 1] = relu6_bf16x2(__uint_as_float(v[4 * j + 2]) + bb.z, __uint_as_float(v[4 * j + 3]) + bb.w);
                    }
                }
                if (threadIdx.x == 64) TCS_TR(3, d, 1);
                mbar_wait_backoff(bar(TcsBars::a_empty, ai), (use & 1u) ^ 1u, TCS_SLEEP_CONVERT);       // the pointwise MMAs have read the previous content
                if (threadIdx.x == 64) TCS_TR(3, d, 2);
                tc_fence_after();
                tcs_st32(tmem + lane_off + TCS_A_COL + (uint32_t)(ai * 32), pk);
                tcs_st_wait();
                tc_fence_before();
                mbar_arrive(bar(TcsBars::a_full, ai));
                if (threadIdx.x == 64) TCS_TR(3, d, 3);
            }
    } else if (warp < 6 + TCS_EPI_WARPS) {
        // ===================== epilogue =====================
        const int ew = warp - 6, quad = warp & 3, half = ew >> 2;
        const uint32_t lane_off = (uint32_t)(quad * 32) << 16;
        const uint32_t stg = base + g.off_stg + (uint32_t)ew * TCS_STG_BYTES;
        const uint32_t spwb = base + g.off_pwb;
        const int slabs = g.nc / 32;
        int item = 0;
        for (long long u = blockIdx.x; u < g.units; u += ustride, ++item) {
            const int img = (int)(u / per_img), rem = (int)(u - (long long)img * per_img);
            const int band = rem / g.chunks, chunk = rem - band * g.chunks;
            long long pix[4];                                     // element offset of the pixel this lane stores in pass i, or -1
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const uint32_t q = (uint32_t)(chunk * 128 + quad * 32 + i * 8 + (lane >> 2));
                const int ty = (int)__umulhi(q, g.magic_wp), tx = (int)q - ty * g.wp;
                const int gx = band * g.tw + tx;
                pix[i] = (tx < g.tw && gx < g.w && ty < g.h) ? (((long long)img * g.h + ty) * g.w + gx) * g.nc : -1;
            }
            mbar_wait_backoff(bar(TcsBars::tfull, 0), (uint32_t)item & 1u, TCS_SLEEP_EPI);
            if (threadIdx.x == 192) TCS_TR(5, item, 0);
            tc_fence_after();
            for (int sl = half; sl < slabs; sl += 2) {
                uint32_t v[32];
                tc_ld32(tmem + lane_off + (uint32_t)(sl * 32), v);
                tc_ld_wait();
                if (sl + 2 >= slabs) {                        // this warp's last read of the accumulator
                    tc_fence_before();
                    mbar_arrive(bar(TcsBars::tempty, 0));
                    if (threadIdx.x == 192) TCS_TR(5, item, 1);
                }
                const uint32_t bcol = spwb + (uint32_t)(sl * 32) * 4u;
                const uint32_t row = stg + (uint32_t)lane * 64u;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float4 b0 = tcs_lds_f4(bcol + (uint32_t)j * 32u), b1 = tcs_lds_f4(bcol + (uint32_t)j * 32u + 16u);
                    st_shared_v4(row + (uint32_t)((j ^ ((lane >> 1) & 3)) * 16),
                                 relu6_bf16x2(__uint_as_float(v[8 * j]) + b0.x, __uint_as_float(v[8 * j + 1]) + b0.y),
                                 relu6_bf16x2(__uint_as_float(v[8 * j + 2]) + b0.z, __uint_as_float(v[8 * j + 3]) + b0.w),
                                 relu6_bf16x2(__uint_as_float(v[8 * j + 4]) + b1.x, __uint_as_float(v[8 * j + 5]) + b1.y),
                                 relu6_bf16x2(__uint_as_float(v[8 * j + 6]) + b1.z, __uint_as_float(v[8 * j + 7]) + b1.w));
                }
                __syncwarp();
                const int ccol = sl * 32 + (lane & 3) * 8;
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int r = i * 8 + (lane >> 2);
                    const uint4 val = ld_shared_v4(stg + (uint32_t)r * 64u + (uint32_t)(((lane & 3) ^ ((r >> 1) & 3)) * 16));
                    if (pix[i] >= 0) tcs_stg_v4(y + pix[i] + ccol, val);
                }
                __syncwarp();
            }
            if (threadIdx.x == 192) TCS_TR(5, item, 2);
        }
    } else if (warp == 14) {
        // ===================== diagonal weight tiles =====================
        // element idx = lane + 32 i (i < 18): tap t = i >> 1, group gq = 2 (i & 1) + (lane >> 4), row n = lane & 15
        const int n = lane & 15, gq0 = lane >> 4;
        const uint32_t sdww = base + g.off_dww;
        const uint32_t dst_e = (uint32_t)(n * 128 + (((gq0 * 2 + (n >> 3)) ^ (n & 7)) * 16) + (n & 7) * 2);
        const uint32_t dst_o = (uint32_t)(n * 128 + ((((gq0 + 2) * 2 + (n >> 3)) ^ (n & 7)) * 16) + (n & 7) * 2);
        const uint32_t src_l = (uint32_t)(gq0 * 16 + n) * 2u;
        int d = 0;
        for (int i = 0; i < my_units; ++i)
            for (int kb = 0; kb < g.kblocks; ++kb, ++d) {
                const int db = d & 1;
                mbar_wait_backoff(bar(TcsBars::diag_empty, db), ((uint32_t)(d >> 1) & 1u) ^ 1u, TCS_SLEEP_DIAG);
                if (lane == 0) TCS_TR(4, d, 0);
                if (g.kblocks > 2 || d < 2) {                      // with <= 2 k-blocks each buffer keeps its k-block for good
                    const uint32_t dst = d_addr(db);
                    uint32_t src = sdww + src_l + (uint32_t)((g.kblocks == 1 ? 0 : kb) * 64) * 2u;
                    uint32_t vals[18];
#pragma unroll
                    for (int t = 0; t < 9; ++t) {
                        vals[2 * t] = tcs_lds_u16(src);
                        vals[2 * t + 1] = tcs_lds_u16(src + 64u);
                        src += (uint32_t)g.k * 2u;
                    }
#pragma unroll
                    for (int t = 0; t < 9; ++t) {
                        tcs_sts_u16(dst + (uint32_t)t * 2048u + dst_e, vals[2 * t]);
                        tcs_sts_u16(dst + (uint32_t)t * 2048u + dst_o, vals[2 * t + 1]);
                    }
                    fence_async_smem();
                }
                __syncwarp();
                if (lane == 0) {
                    mbar_arrive(bar(TcsBars::diag_full, db));
                    TCS_TR(4, d, 1);
                }
            }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
}

// ---- host side ---------------------------------------------------------------------------------------------
// Which blocks take this path: 256 -> 256, stride 1, dilation 1 or 2.  Measured on B200 (profiles/r01_v9_septc_experiment.md):
// a tap MMA costs 32 + N/4 cycles (operand fetch: every M128 x N16 x K16 MMA re-reads 4 KB of patch from shared memory), so the
// depthwise is no cheaper here than on the CUDA cores and it serialises with the pointwise MMAs on the one tensor pipe.  It wins
// where the CUDA-core kernel is at its weakest and this one at its best -- 256 -> 256 blocks (one 256-column accumulator, A
// ring): 0.178 vs 0.203 ms on the dilated blocks of model 50 at OS8 (C3), 0.104 vs 0.107 ms on block 5 of model 101 (C2) -- and
// loses on the other widths it was tried at (128 -> 128: 0.199 vs 0.186 ms, 512 -> 512: 0.096 vs 0.073 ms).
bool septc_supported(int k, int nc, int stride, int dil) { return stride == 1 && (dil == 1 || dil == 2) && k == 256 && nc == 256; }

int septc_geometry(SepTcOp *op, int n, int h, int wd, int k, int nc, int dil) {
    PN_CHECK_ARG(septc_supported(k, nc, 1, dil), "septc: unsupported block");
    TcsGeom g;
    memset(&g, 0, sizeof(g));
    g.k = k; g.nc = nc; g.h = h; g.w = wd; g.n_img = n; g.dil = dil;
    g.kblocks = k / 64;
    g.w_stage_bytes = (unsigned)nc * 128u;
    const unsigned table_bytes = (unsigned)((9 * k * 2 + 15) / 16 * 16 + k * 4 + nc * 4);
    const long long fixed = 1024 + 2LL * TCS_DIAG_BYTES + (long long)TCS_EPI_WARPS * TCS_STG_BYTES + table_bytes + TcsBars::total;
    // column bands: pitch wp = tw + 2 dil (one band over the whole width shares the zero gap: wp = w + dil).  Cost per unit in
    // shared-memory cycles (128 B/clk): 9 tap reads of 128 rows + (half) the patch write per k-block, W write + read per pointwise
    // step, + a per-unit overhead; the weights are fitted to band sweeps on the C2 / C3 blocks: wide bands win.
    double best = 1e30;
    for (int bands = 1; bands <= 16; ++bands) {
        const int tw = ceil_div(wd, bands);
        if (bands > 1 && ceil_div(wd, tw) != bands) continue;
        const int wp = bands == 1 ? wd + dil : tw + 2 * dil;
        if (wp > 256) continue;
        const int rows_box = ceil_div(wp - 1 + 127 + 2 * dil * wp + 2 * dil + 1, wp);
        if (rows_box > 256) continue;
        const long long patch = (long long)rows_box * wp * 128;
        const long long stage = (patch + 1023) / 1024 * 1024;
        if (fixed + 2 * stage + 2LL * g.w_stage_bytes > TCS_SMEM_MAX) continue;
        const int chunks = ceil_div((h - 1) * wp + tw, 128);
        const double per_unit = g.kblocks * (1152.0 + patch / 256.0) + g.kblocks * (2.0 * g.w_stage_bytes / 128.0) + 600.0;
        const double cost = (double)bands * chunks * per_unit;
        // (measured: fewer, wider bands win even when they leave room for two patch stages only -- C3 0.178 ms with 4 bands / 2
        // stages against 0.193 ms with 7 bands / 3 stages -- so the stage count is not part of the cost)
        if (cost < best) {
            best = cost;
            g.bands = bands; g.tw = tw; g.wp = wp; g.rows_box = rows_box; g.chunks = chunks;
            g.patch_bytes = (unsigned)patch; g.patch_stage_bytes = (unsigned)stage;
        }
    }
    PN_CHECK_ARG(best < 1e30, "septc: no band layout fits (h %d w %d cin %d cout %d dilation %d)", h, wd, k, nc, dil);
    // the last row any tap MMA reads (chunk start at most wp - 1 rows into the box, + the bottom-right tap, + 128 rows) lies
    // inside the stage, so no descriptor ever points past the patch it belongs to
    PN_CHECK_ARG((long long)(g.wp - 1 + 2 * dil * g.wp + 2 * dil + 128) * 128 <= (long long)g.patch_stage_bytes,
                 "septc: internal error, tap view exceeds the patch stage");
    g.magic_wp = (unsigned)((0x100000000ull + (unsigned)g.wp - 1) / (unsigned)g.wp);
    PN_CHECK_ARG((long long)g.chunks * 128 + 128 < (long long)(0x100000000ull / (unsigned)g.wp), "septc: image too large for the pitch division");
    g.units = (long long)n * g.bands * g.chunks;
    // stages: a third patch stage first (the TMA latency exceeds one depthwise step), then W stages, then a fourth patch stage
    g.p_stages = 2; g.w_stages = 2;
    auto total = [&](int ps, int ws) { return fixed + (long long)ps * g.patch_stage_bytes + (long long)ws * g.w_stage_bytes; };
    if (total(3, 2) <= TCS_SMEM_MAX) g.p_stages = 3;
    while (g.w_stages < TCS_MAX_W && total(g.p_stages, g.w_stages + 1) <= TCS_SMEM_MAX) ++g.w_stages;
    if (g.p_stages == 3 && total(4, g.w_stages) <= TCS_SMEM_MAX) g.p_stages = 4;
    g.off_diag = (unsigned)g.w_stages * g.w_stage_bytes;
    g.off_patch = g.off_diag + 2u * TCS_DIAG_BYTES;
    g.off_stg = g.off_patch + (unsigned)g.p_stages * g.patch_stage_bytes;
    g.off_dww = g.off_stg + (unsigned)TCS_EPI_WARPS * TCS_STG_BYTES;
    g.off_dwb = g.off_dww + (unsigned)((9 * k * 2 + 15) / 16 * 16);
    g.off_pwb = g.off_dwb + (unsigned)k * 4u;
    g.off_bar = g.off_pwb + (unsigned)nc * 4u;
    op->smem_bytes = (int)(g.off_bar + TcsBars::total + 1024);
    PN_CHECK_ARG(op->smem_bytes <= TCS_SMEM_MAX, "septc: internal smem accounting error (%d)", op->smem_bytes);
    static_assert(sizeof(TcsGeom) <= sizeof(op->geom), "SepTcOp::geom too small");
    memcpy(op->geom, &g, sizeof(g));
    return PN_OK;
}

int septc_prepare(SepTcOp *op, const void *x, const void *pw_w, int n, int h, int wd, int k, int nc, int dil) {
    int rc = septc_geometry(op, n, h, wd, k, nc, dil);
    if (rc != PN_OK) return rc;
    TcsGeom g;
    memcpy(&g, op->geom, sizeof(g));
    {   // input patches: (C, W, H, N) bf16, box [64, wp, rows_box, 1], 128B swizzle, OOB -> 0 (== zero padding)
        const uint64_t dims[4] = {(uint64_t)k, (uint64_t)wd, (uint64_t)h, (uint64_t)n};
        const uint64_t strides[3] = {(uint64_t)k * 2, (uint64_t)wd * k * 2, (uint64_t)h * wd * k * 2};
        const uint32_t box[4] = {64u, (uint32_t)g.wp, (uint32_t)g.rows_box, 1u};
        if ((rc = encode_tmap(op->tmap_x, x, 2, 4, dims, strides, box, 3)) != PN_OK) return rc;
    }
    {   // pointwise weights [Nc, K] bf16, box [64, Nc], 128B swizzle
        const uint64_t dims[2] = {(uint64_t)k, (uint64_t)nc};
        const uint64_t strides[1] = {(uint64_t)k * 2};
        const uint32_t box[2] = {64u, (uint32_t)nc};
        if ((rc = encode_tmap(op->tmap_w, pw_w, 2, 2, dims, strides, box, 3)) != PN_OK) return rc;
    }
    return PN_OK;
}

int septc_launch(const SepTcOp *op, const float *dw_w, const float *dw_b, const float *pw_b, void *y, cudaStream_t st) {
    static DeviceOnce once;
    const int dev = current_device();
    TcsGeom g;
    memcpy(&g, op->geom, sizeof(g));
    if (!once.get(dev)) {
        PN_CHECK_CUDA(cudaFuncSetAttribute(septc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TCS_SMEM_MAX));
        once.set(dev, 1);
    }
    const long long sms = num_sms();
    const int grid = (int)(g.units < sms ? g.units : sms);
    PN_CHECK_CUDA(launch_pdl(septc_kernel, dim3((unsigned)grid), dim3(TCS_THREADS), (size_t)op->smem_bytes, st,
                             *reinterpret_cast<const CUtensorMap *>(op->tmap_x), *reinterpret_cast<const CUtensorMap *>(op->tmap_w), dw_w,
                             dw_b, pw_b, reinterpret_cast<__nv_bfloat16 *>(y), g));
    return PN_OK;
}

void septc_describe(const SepTcOp *op, char *out, size_t cap) {
    TcsGeom g;
    memcpy(&g, op->geom, sizeof(g));
    snprintf(out, cap, "tensor-pipe depthwise: bands %d x %d cols pitch %d box rows %d chunks %d kblocks %d stages p%d w%d smem %d units %lld",
             g.bands, g.tw, g.wp, g.rows_box, g.chunks, g.kblocks, g.p_stages, g.w_stages, op->smem_bytes, g.units);
}

}  // namespace pn

#ifdef PN_TCS_TRACE
// diagnostics build: trace buffer = 6 roles x cap steps x 4 stamps (int64), zero-filled by the caller; (nullptr, 0) turns it off
extern "C" int pn_debug_tcs_trace(long long *buf, int cap) {
    if (cudaMemcpyToSymbol(pn::g_tcs_trace, &buf, sizeof(buf)) != cudaSuccess) return -2;
    if (cudaMemcpyToSymbol(pn::g_tcs_trace_cap, &cap, sizeof(cap)) != cudaSuccess) return -2;
    return 0;
}
#endif
