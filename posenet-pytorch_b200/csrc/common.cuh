// Shared host/device helpers for libposenet_b200 (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <atomic>

#include "../../include/posenet_b200.h"

namespace pn {

// ---- error plumbing -------------------------------------------------------------------------
void set_error(const char *fmt, ...);

#define PN_CHECK_ARG(cond, ...)           \
    do {                                  \
        if (!(cond)) {                    \
            pn::set_error(__VA_ARGS__);   \
            return PN_ERR_ARG;            \
        }                                 \
    } while (0)

#define PN_CHECK_CUDA(expr)                                                                   \
    do {                                                                                      \
        cudaError_t _e = (expr);                                                              \
        if (_e != cudaSuccess) {                                                              \
            pn::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return PN_ERR_CUDA;                                                               \
        }                                                                                     \
    } while (0)

#define PN_CHECK_LAUNCH() PN_CHECK_CUDA(cudaGetLastError())

inline cudaStream_t as_stream(pn_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

// Kernel launch with programmatic stream serialization (PDL): the persistent kernels of consecutive layers overlap the
// prologue of layer i+1 (barrier init, TMEM allocation, weight staging) with the tail of layer i.  Every kernel launched
// this way executes griddepcontrol.wait (pdl_wait, ptx.cuh) before it touches activations.  PN_NO_PDL=1 disables it.
bool pdl_enabled();
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args &&...args) {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}
inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
int current_device();   // cudaGetDevice (0 when the query fails)
int num_sms();          // SM count of the CURRENT device

// One-time setup per DEVICE: cudaFuncSetAttribute(MaxDynamicSharedMemorySize) and occupancy queries apply to the current
// device only, so a process that drives several GPUs must repeat them on each.  Usage:
//     static DeviceOnce once;  const int dev = current_device();
//     if (once.get(dev) < wanted) { ...setup on the current device...;  once.set(dev, wanted); }
// Racing threads at worst both run the (idempotent) setup.
constexpr int PN_MAX_DEVICES = 64;
struct DeviceOnce {
    std::atomic<int> v[PN_MAX_DEVICES];
    int get(int dev) const { return dev >= 0 && dev < PN_MAX_DEVICES ? v[dev].load(std::memory_order_acquire) : 0; }
    void set(int dev, int value) { if (dev >= 0 && dev < PN_MAX_DEVICES) v[dev].store(value, std::memory_order_release); }
};

// ---- shared epilogue description for both GEMM paths -------------------------------------------
// EPI_RELU6: y[m, n] = clamp(acc + bias[n], 0, 6) stored row-major [M, N] in the activation dtype.
// EPI_HEADS: the 115 head channels scattered to four fp32 NCHW tensors, sigmoid on the heatmap.
enum { EPI_RELU6 = 0, EPI_HEADS = 1 };

struct EpiParams {
    const float *bias;
    void *y;        // EPI_RELU6
    float *heat, *off, *fwd, *bwd;  // EPI_HEADS
    int hw;         // EPI_HEADS: pixels per image
};

__device__ __forceinline__ float relu6f(float v) { return fminf(fmaxf(v, 0.f), 6.f); }

// Head column -> (tensor, channel).  Layout of the packed head rows: heat 0..16, offset 17..50,
// displacement_fwd 51..82, displacement_bwd 83..114 (mobilenet_v1.py:151-154).
__device__ __forceinline__ void store_head(const EpiParams &ep, int m, int col, float v) {
    int img = m / ep.hw;
    int p = m - img * ep.hw;
    if (col < 17) {
        ep.heat[((size_t)img * 17 + col) * ep.hw + p] = 1.f / (1.f + expf(-v));   // mobilenet_v1.py:158
    } else if (col < 51) {
        ep.off[((size_t)img * 34 + (col - 17)) * ep.hw + p] = v;
    } else if (col < 83) {
        ep.fwd[((size_t)img * 32 + (col - 51)) * ep.hw + p] = v;
    } else if (col < 115) {
        ep.bwd[((size_t)img * 32 + (col - 83)) * ep.hw + p] = v;
    }
}

// ---- typed activation load/store (fp32 | bf16), 8 channels at a time -------------------------
template <typename T> struct Vec8;
template <> struct Vec8<float> {
    static __device__ __forceinline__ void load(const float *p, float (&v)[8]) {
        float4 a = *reinterpret_cast<const float4 *>(p);
        float4 b = *reinterpret_cast<const float4 *>(p + 4);
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    }
    static __device__ __forceinline__ void store(float *p, const float (&v)[8]) {
        *reinterpret_cast<float4 *>(p) = make_float4(v[0], v[1], v[2], v[3]);
        *reinterpret_cast<float4 *>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
    }
};
template <> struct Vec8<__nv_bfloat16> {
    static __device__ __forceinline__ void load(const __nv_bfloat16 *p, float (&v)[8]) {
        uint4 r = *reinterpret_cast<const uint4 *>(p);
        const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {   // bf16 -> f32 is a 16-bit shift
            v[2 * i] = __uint_as_float(w[i] << 16);
            v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
        }
    }
    static __device__ __forceinline__ void store(__nv_bfloat16 *p, const float (&v)[8]) {
        uint32_t w[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
            w[i] = *reinterpret_cast<uint32_t *>(&h);
        }
        *reinterpret_cast<uint4 *>(p) = make_uint4(w[0], w[1], w[2], w[3]);
    }
};

// ---- launchers implemented one per .cu file ----------------------------------------------------
int launch_preprocess(const uint8_t *src, int n, int sh, int sw, int dh, int dw, float *dst, cudaStream_t s);
int launch_resize_u8(const uint8_t *src, int n, int sh, int sw, int dh, int dw, uint8_t *dst, cudaStream_t s);
int launch_stem(const void *x, bool x_is_u8, const float *w, const float *b, void *y, int n, int h, int wd,
                int cout, int stride, int out_dtype, cudaStream_t s);
int launch_dwconv(const void *x, const float *w, const float *b, void *y, int n, int h, int wd, int c,
                  int stride, int dilation, int dtype, cudaStream_t s);
// stride-1 bf16 depthwise as warp-autonomous strips (dwwarp.cu)
struct DwWarpOp {
    alignas(64) unsigned char tmap_x[128];
    alignas(8) unsigned char geom[64];
    int dil;
};
bool dwwarp_supported(int c, int stride, int dil, int dtype);
int dwwarp_prepare(DwWarpOp *op, const void *x, int n, int h, int wd, int c, int dil);
int dwwarp_launch(const DwWarpOp *op, const float *w, const float *b, void *y, cudaStream_t s);

// depthwise op bound to one input buffer: tensor map + tile geometry are computed once (per plan, or per call)
struct DwOp {
    alignas(64) unsigned char tmap[128];
    alignas(8) unsigned char geom[128];
    const void *x;
    int n, h, w, c, stride, dil, dtype, ho, wo;
    bool use_tma;
    bool warp_kind;          // stride 1, dilation 1 / 2, bf16: the strip kernel of dwwarp.cu
    DwWarpOp warp;
};
int dw_prepare(DwOp *op, const void *x, int n, int h, int wd, int c, int stride, int dil, int dtype);
int dw_launch(const DwOp *op, const float *w, const float *b, void *y, cudaStream_t s);
int launch_gemm_simt(const float *a, const float *w, int m, int k, int n, int epi, const EpiParams &ep,
                     cudaStream_t s);

// tcgen05 path: tensor maps are encoded once (per plan, or per standalone call) then reused.
struct GemmTc {
    alignas(64) unsigned char tmap_a[128];
    alignas(64) unsigned char tmap_b[128];
    alignas(64) unsigned char tmap_c[128];   // output map (TMA-store epilogue), bound to one output buffer
    int m, k, n, block_n, epi;
};
int gemm_tc_prepare(GemmTc *g, const void *a, const void *w, void *y, int m, int k, int n, int epi);
int gemm_tc_launch(const GemmTc *g, const EpiParams &ep, cudaStream_t s);

// narrow fused block (cin <= 32, cout <= 64, dilation 1; stride 1, or stride 2 with cin > 16): warp-autonomous kernel (sepwarp.cu)
struct SepWarpOp {
    alignas(64) unsigned char tmap_x[128];
    alignas(8) unsigned char geom[64];
};
bool sepwarp_supported(int k, int nc, int stride, int dil);
int sepwarp_geometry(SepWarpOp *op, int n, int h, int wd, int k, int nc, int stride);
int sepwarp_prepare(SepWarpOp *op, const void *x, int n, int h, int wd, int k, int nc, int stride);
int sepwarp_launch(const SepWarpOp *op, const float *dw_w, const float *dw_b, const void *pw_w, const float *pw_b, void *y,
                   cudaStream_t s);
void sepwarp_describe(const SepWarpOp *op, char *out, size_t cap);

// fused block with the depthwise on the tensor pipe (septc.cu): stride 1, dilation 1 / 2, cin = cout = 256
struct SepTcOp {
    alignas(64) unsigned char tmap_x[128];
    alignas(64) unsigned char tmap_w[128];
    alignas(8) unsigned char geom[256];
    int smem_bytes;
};
bool septc_supported(int k, int nc, int stride, int dil);   // the 256 -> 256 blocks at stride 1, dilation 1 or 2 (measured)
int septc_geometry(SepTcOp *op, int n, int h, int wd, int k, int nc, int dil);
int septc_prepare(SepTcOp *op, const void *x, const void *pw_w, int n, int h, int wd, int k, int nc, int dil);
int septc_launch(const SepTcOp *op, const float *dw_w, const float *dw_b, const float *pw_b, void *y, cudaStream_t s);
void septc_describe(const SepTcOp *op, char *out, size_t cap);

// fused SeperableConv block (depthwise -> pointwise in one kernel, sepconv.cu); bf16 only
struct SepOp {
    alignas(64) unsigned char tmap_x[128];
    alignas(64) unsigned char tmap_dww[128];
    alignas(64) unsigned char tmap_dwb[128];
    alignas(64) unsigned char tmap_w[128];
    alignas(64) unsigned char tmap_y[128];
    alignas(8) unsigned char geom[640];
    int smem_bytes, cb, stride, dil, ho, wo, n, h, w, k, nc;
    // narrow blocks run the warp-autonomous kernel instead (warp_kind): it takes plain pointers, kept here for the launch
    bool warp_kind;
    SepWarpOp warp;
    bool tc_kind;            // depthwise on the tensor pipe (septc.cu)
    SepTcOp tc;
    const float *dw_w, *dw_b;
    const void *pw_w;
    void *y;
};
bool sep_supported(int k, int nc, int stride, int dil);
bool sep_fuse_recommended(int k, int nc, int stride, int dil);
int sep_geometry(SepOp *op, int n, int h, int wd, int k, int nc, int stride, int dil);
int sep_prepare(SepOp *op, const void *x, const float *dw_w, const float *dw_b, const void *pw_w, void *y, int n, int h,
                int wd, int k, int nc, int stride, int dil);
int sep_launch(const SepOp *op, const float *pw_bias, cudaStream_t s);
void sep_describe(const SepOp *op, char *out, size_t cap);

}  // namespace pn
