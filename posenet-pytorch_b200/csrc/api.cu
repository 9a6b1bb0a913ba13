// C ABI glue: error strings, per-op entry points and the whole-network plan (include/posenet_b200.h).
#include <cuda.h>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <new>
#include <vector>

#include "common.cuh"

namespace pn {

static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

bool pdl_enabled() {
    static int on = -1;
    if (on < 0) on = getenv("PN_NO_PDL") == nullptr ? 1 : 0;
    return on == 1;
}

int current_device() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { (void)cudaGetLastError(); dev = 0; }
    return dev;
}

int num_sms() {
    static DeviceOnce cache;                      // per device: a mixed box must not size grids by device 0's SM count
    const int dev = current_device();
    int sms = cache.get(dev);
    if (sms <= 0) {
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
        cache.set(dev, sms);
    }
    return sms;
}

static size_t esize(int dtype) { return dtype == PN_BF16 ? 2 : 4; }

static int conv_out(int in, int stride, int dil) {
    const int pad = ((stride - 1) + dil * 2) / 2;            // mobilenet_v1.py:42-44 with k = 3
    return (in + 2 * pad - 2 * dil - 1) / stride + 1;
}

}  // namespace pn

using namespace pn;

struct pn_plan {
    pn_net_desc d;
    void *buf[2];
    int out_h, out_w;
    struct Step {
        int h_in, w_in, h_out, w_out;
        bool fused;         // bf16: the whole block is one sepconv launch
        GemmTc tc;          // bf16 only
        DwOp dw;
        SepOp sep;
    } steps[16];
    GemmTc head_tc;
    int launches;
    char names[40][12];
};

extern "C" {

int pn_abi_version(void) { return PN_ABI_VERSION; }
const char *pn_last_error_string(void) { return g_err; }

int pn_device_check(void) {
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) {
        (void)cudaGetLastError();
        set_error("no CUDA device visible");
        return PN_ERR_NO_DEVICE;
    }
    int dev = 0, major = 0, minor = 0;
    PN_CHECK_CUDA(cudaGetDevice(&dev));
    PN_CHECK_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
    PN_CHECK_CUDA(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev));
    if (major != 10) {
        set_error("device %d is sm_%d%d; libposenet_b200 is built for sm_100a only", dev, major, minor);
        return PN_ERR_UNSUPPORTED;
    }
    return PN_OK;
}

int pn_preprocess_u8(const uint8_t *src, int n, int src_h, int src_w, int dst_h, int dst_w, float *dst,
                     pn_stream_t stream) {
    return launch_preprocess(src, n, src_h, src_w, dst_h, dst_w, dst, as_stream(stream));
}

int pn_resize_u8(const uint8_t *src, int n, int src_h, int src_w, int dst_h, int dst_w, uint8_t *dst, pn_stream_t stream) {
    return launch_resize_u8(src, n, src_h, src_w, dst_h, dst_w, dst, as_stream(stream));
}

int pn_stem_conv(const float *x, const float *w, const float *bias, void *y, int n, int h, int wd, int cout,
                 int stride, int out_dtype, pn_stream_t stream) {
    return launch_stem(x, false, w, bias, y, n, h, wd, cout, stride, out_dtype, as_stream(stream));
}

int pn_stem_conv_u8(const uint8_t *img, const float *w, const float *bias, void *y, int n, int h, int wd, int cout,
                    int stride, int out_dtype, pn_stream_t stream) {
    return launch_stem(img, true, w, bias, y, n, h, wd, cout, stride, out_dtype, as_stream(stream));
}

int pn_dwconv3x3(const void *x, const float *w, const float *bias, void *y, int n, int h, int wd, int c, int stride,
                 int dilation, int dtype, pn_stream_t stream) {
    return launch_dwconv(x, w, bias, y, n, h, wd, c, stride, dilation, dtype, as_stream(stream));
}

int pn_pwconv_gemm(const void *a, const void *w, const float *bias, void *y, int m, int k, int n, int dtype,
                   pn_stream_t stream) {
    PN_CHECK_ARG(bias && y, "pn_pwconv_gemm: null pointer");
    EpiParams ep = {};
    ep.bias = bias;
    ep.y = y;
    if (dtype == PN_F32) return launch_gemm_simt((const float *)a, (const float *)w, m, k, n, EPI_RELU6, ep, as_stream(stream));
    PN_CHECK_ARG(dtype == PN_BF16, "pn_pwconv_gemm: bad dtype %d", dtype);
    GemmTc g;
    int rc = gemm_tc_prepare(&g, a, w, y, m, k, n, EPI_RELU6);
    if (rc != PN_OK) return rc;
    return gemm_tc_launch(&g, ep, as_stream(stream));
}

int pn_sepconv_block(const void *x, const float *dw_w, const float *dw_b, const void *pw_w, const float *pw_b, void *y, int n,
                     int h, int wd, int cin, int cout, int stride, int dilation, pn_stream_t stream) {
    SepOp op;
    int rc = sep_prepare(&op, x, dw_w, dw_b, pw_w, y, n, h, wd, cin, cout, stride, dilation);
    if (rc != PN_OK) return rc;
    return sep_launch(&op, pw_b, as_stream(stream));
}

int pn_sepconv_describe(int n, int h, int wd, int cin, int cout, int stride, int dilation, char *out_host, int capacity) {
    PN_CHECK_ARG(out_host && capacity > 0, "pn_sepconv_describe: null buffer");
    SepOp op;
    int rc = sep_geometry(&op, n, h, wd, cin, cout, stride, dilation);
    if (rc != PN_OK) return rc;
    sep_describe(&op, out_host, (size_t)capacity);
    return PN_OK;
}

int pn_heads_gemm(const void *a, const void *w, const float *bias, float *heat, float *off, float *fwd, float *bwd,
                  int n_img, int hw, int k, int dtype, pn_stream_t stream) {
    PN_CHECK_ARG(bias && heat && off && fwd && bwd && n_img > 0 && hw > 0, "pn_heads_gemm: bad argument");
    EpiParams ep = {};
    ep.bias = bias;
    ep.heat = heat; ep.off = off; ep.fwd = fwd; ep.bwd = bwd;
    ep.hw = hw;
    const int m = n_img * hw;
    if (dtype == PN_F32)
        return launch_gemm_simt((const float *)a, (const float *)w, m, k, PN_HEAD_ROWS, EPI_HEADS, ep, as_stream(stream));
    PN_CHECK_ARG(dtype == PN_BF16, "pn_heads_gemm: bad dtype %d", dtype);
    GemmTc g;
    int rc = gemm_tc_prepare(&g, a, w, nullptr, m, k, PN_HEAD_ROWS, EPI_HEADS);
    if (rc != PN_OK) return rc;
    return gemm_tc_launch(&g, ep, as_stream(stream));
}

// ---- plan ------------------------------------------------------------------------------------------
static int plan_shapes(const pn_net_desc *d, size_t *arena_bytes, int *out_h, int *out_w, pn_plan *plan) {
    PN_CHECK_ARG(d, "pn_plan: null descriptor");
    PN_CHECK_ARG(d->dtype == PN_F32 || d->dtype == PN_BF16, "pn_plan: bad dtype %d", d->dtype);
    PN_CHECK_ARG(d->n > 0 && d->h > 0 && d->w > 0, "pn_plan: bad input shape %d x %d x %d", d->n, d->h, d->w);
    PN_CHECK_ARG(d->num_layers >= 1 && d->num_layers <= 16, "pn_plan: bad layer count %d", d->num_layers);
    int h = d->h, w = d->w;
    size_t max_elems = 0;
    for (int i = 0; i < d->num_layers; ++i) {
        const pn_layer &L = d->layers[i];
        PN_CHECK_ARG(L.cout % 8 == 0 && (i == 0 || L.cin % 8 == 0), "pn_plan: layer %d channels %d->%d not multiples of 8", i,
                     L.cin, L.cout);
        PN_CHECK_ARG(i == 0 ? L.cin == 3 : L.cin == d->layers[i - 1].cout, "pn_plan: layer %d cin mismatch", i);
        const int ho = conv_out(h, L.stride, L.dilation), wo = conv_out(w, L.stride, L.dilation);
        PN_CHECK_ARG(ho > 0 && wo > 0, "pn_plan: layer %d produces an empty map", i);
        if (plan) {
            plan->steps[i].h_in = h; plan->steps[i].w_in = w;
            plan->steps[i].h_out = ho; plan->steps[i].w_out = wo;
        }
        const size_t m = (size_t)d->n * ho * wo;
        PN_CHECK_ARG(m < (1ull << 31), "pn_plan: layer %d has too many pixels", i);
        const size_t cmax = L.cin > L.cout ? L.cin : L.cout;
        if (m * cmax > max_elems) max_elems = m * cmax;
        h = ho; w = wo;
    }
    if (arena_bytes) *arena_bytes = 2 * ((max_elems * esize(d->dtype) + 1023) & ~(size_t)1023);
    if (out_h) *out_h = h;
    if (out_w) *out_w = w;
    return PN_OK;
}

int pn_plan_query(const pn_net_desc *desc, size_t *arena_bytes, int *out_h, int *out_w) {
    return plan_shapes(desc, arena_bytes, out_h, out_w, nullptr);
}

int pn_plan_create(const pn_net_desc *desc, void *arena, size_t arena_bytes, pn_plan **out) {
    PN_CHECK_ARG(out && arena, "pn_plan_create: null pointer");
    *out = nullptr;
    pn_plan *p = new (std::nothrow) pn_plan();
    PN_CHECK_ARG(p, "pn_plan_create: out of host memory");
    size_t need = 0;
    int rc = plan_shapes(desc, &need, &p->out_h, &p->out_w, p);
    if (rc == PN_OK && (arena_bytes < need || ((uintptr_t)arena & 1023))) {
        set_error("pn_plan_create: arena must be 1024-byte aligned and >= %zu bytes (got %zu)", need, arena_bytes);
        rc = PN_ERR_ARG;
    }
    if (rc != PN_OK) { delete p; return rc; }
    p->d = *desc;
    p->buf[0] = arena;
    p->buf[1] = (char *)arena + need / 2;
    p->launches = 0;
    // Buffer schedule: the current activation lives in buf[cur] (stem -> buf0).  A fused block reads buf[cur] and
    // writes buf[cur^1]; an unfused block runs dw buf[cur] -> buf[cur^1], pw buf[cur^1] -> buf[cur].
    int cur = 0;
    for (int i = 0; i < desc->num_layers; ++i) {
        const pn_layer &L = desc->layers[i];
        pn_plan::Step &S = p->steps[i];
        if (!(L.pw_w && L.pw_b && (i == 0 || (L.dw_w && L.dw_b)))) {
            set_error("pn_plan_create: layer %d has null weights", i);
            delete p;
            return PN_ERR_ARG;
        }
        if (i == 0) {
            snprintf(p->names[p->launches++], sizeof(p->names[0]), "stem");
            continue;
        }
        // Fuse a block when the depthwise work is done once per tile (sep_fuse_recommended)
        S.fused = desc->dtype == PN_BF16 && !(desc->flags & PN_PLAN_UNFUSED) && sep_fuse_recommended(L.cin, L.cout, L.stride, L.dilation);
        if (S.fused) {
            rc = sep_prepare(&S.sep, p->buf[cur], L.dw_w, L.dw_b, L.pw_w, p->buf[cur ^ 1], desc->n, S.h_in, S.w_in, L.cin, L.cout,
                             L.stride, L.dilation);
            if (rc != PN_OK) { delete p; return rc; }
            snprintf(p->names[p->launches++], sizeof(p->names[0]), "sep%d", i);
            cur ^= 1;
            continue;
        }
        rc = dw_prepare(&S.dw, p->buf[cur], desc->n, S.h_in, S.w_in, L.cin, L.stride, L.dilation, desc->dtype);
        if (rc != PN_OK) { delete p; return rc; }
        if (desc->dtype == PN_BF16) {
            const int m = desc->n * S.h_out * S.w_out;
            rc = gemm_tc_prepare(&S.tc, p->buf[cur ^ 1], L.pw_w, p->buf[cur], m, L.cin, L.cout, EPI_RELU6);
            if (rc != PN_OK) { delete p; return rc; }
        }
        snprintf(p->names[p->launches++], sizeof(p->names[0]), "dw%d", i);
        snprintf(p->names[p->launches++], sizeof(p->names[0]), "pw%d", i);
    }
    if (!(desc->head_w && desc->head_b)) {
        set_error("pn_plan_create: null head weights");
        delete p;
        return PN_ERR_ARG;
    }
    if (desc->dtype == PN_BF16) {
        const int m = desc->n * p->out_h * p->out_w;
        rc = gemm_tc_prepare(&p->head_tc, p->buf[cur], desc->head_w, nullptr, m, desc->layers[desc->num_layers - 1].cout, PN_HEAD_ROWS, EPI_HEADS);
        if (rc != PN_OK) { delete p; return rc; }
    }
    snprintf(p->names[p->launches++], sizeof(p->names[0]), "heads");
    *out = p;
    return PN_OK;
}

static int plan_run(pn_plan *p, const void *input, float *heat, float *off, float *fwd, float *bwd, cudaStream_t st,
                    cudaEvent_t *ev /* launches + 1 events or NULL */) {
    const pn_net_desc &d = p->d;
    int rc, li = 0, cur = 0;
#define PN_MARK()                                              \
    do {                                                       \
        if (ev) PN_CHECK_CUDA(cudaEventRecord(ev[li], st));    \
        ++li;                                                  \
    } while (0)
    PN_MARK();
    for (int i = 0; i < d.num_layers; ++i) {
        const pn_layer &L = d.layers[i];
        const pn_plan::Step &S = p->steps[i];
        if (i == 0) {
            rc = launch_stem(input, d.input_u8 != 0, (const float *)L.pw_w, L.pw_b, p->buf[0], d.n, S.h_in, S.w_in, L.cout,
                             L.stride, d.dtype, st);
            if (rc != PN_OK) return rc;
            PN_MARK();
            continue;
        }
        if (S.fused) {
            rc = sep_launch(&S.sep, L.pw_b, st);
            if (rc != PN_OK) return rc;
            PN_MARK();
            cur ^= 1;
            continue;
        }
        rc = dw_launch(&S.dw, L.dw_w, L.dw_b, p->buf[cur ^ 1], st);
        if (rc != PN_OK) return rc;
        PN_MARK();
        EpiParams ep = {};
        ep.bias = L.pw_b;
        ep.y = p->buf[cur];
        const int m = d.n * S.h_out * S.w_out;
        if (d.dtype == PN_BF16)
            rc = gemm_tc_launch(&S.tc, ep, st);
        else
            rc = launch_gemm_simt((const float *)p->buf[cur ^ 1], (const float *)L.pw_w, m, L.cin, L.cout, EPI_RELU6, ep, st);
        if (rc != PN_OK) return rc;
        PN_MARK();
    }
    EpiParams ep = {};
    ep.bias = d.head_b;
    ep.heat = heat; ep.off = off; ep.fwd = fwd; ep.bwd = bwd;
    ep.hw = p->out_h * p->out_w;
    const int m = d.n * ep.hw;
    if (d.dtype == PN_BF16)
        rc = gemm_tc_launch(&p->head_tc, ep, st);
    else
        rc = launch_gemm_simt((const float *)p->buf[cur], (const float *)d.head_w, m, d.layers[d.num_layers - 1].cout, PN_HEAD_ROWS,
                              EPI_HEADS, ep, st);
    if (rc != PN_OK) return rc;
    PN_MARK();
#undef PN_MARK
    return PN_OK;
}

int pn_plan_forward(pn_plan *p, const void *input, float *heat, float *off, float *fwd, float *bwd, pn_stream_t stream) {
    PN_CHECK_ARG(p && input && heat && off && fwd && bwd, "pn_plan_forward: null pointer");
    return plan_run(p, input, heat, off, fwd, bwd, as_stream(stream), nullptr);
}

int pn_plan_profile(pn_plan *p, const void *input, float *heat, float *off, float *fwd, float *bwd, float *ms_host,
                    int capacity, pn_stream_t stream) {
    PN_CHECK_ARG(p && input && heat && off && fwd && bwd && ms_host, "pn_plan_profile: null pointer");
    PN_CHECK_ARG(capacity >= p->launches, "pn_plan_profile: ms_host needs %d entries", p->launches);
    std::vector<cudaEvent_t> ev(p->launches + 1);
    for (auto &e : ev) PN_CHECK_CUDA(cudaEventCreate(&e));
    int rc = plan_run(p, input, heat, off, fwd, bwd, as_stream(stream), ev.data());
    if (rc == PN_OK && cudaStreamSynchronize(as_stream(stream)) != cudaSuccess) {
        set_error("pn_plan_profile: synchronize failed: %s", cudaGetErrorString(cudaGetLastError()));
        rc = PN_ERR_CUDA;
    }
    for (int i = 0; rc == PN_OK && i < p->launches; ++i)
        if (cudaEventElapsedTime(&ms_host[i], ev[i], ev[i + 1]) != cudaSuccess) rc = PN_ERR_CUDA;
    for (auto &e : ev) cudaEventDestroy(e);
    return rc;
}

int pn_plan_num_launches(const pn_plan *plan) { return plan ? plan->launches : 0; }

const char *pn_plan_launch_name(const pn_plan *plan, int i) {
    return (plan && i >= 0 && i < plan->launches) ? plan->names[i] : "";
}

int pn_plan_destroy(pn_plan *plan) {
    delete plan;
    return PN_OK;
}

}  // extern "C"
