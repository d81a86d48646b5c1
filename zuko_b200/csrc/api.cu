// zuko_b200 — C ABI: handles, layer / flow orchestration, workspace carving, row chunking.
// Declarations and reference citations: include/zuko_b200.h.

#include <stdarg.h>
#include <string.h>

#include <algorithm>
#include <mutex>
#include <new>
#include <vector>

#include "api_internal.cuh"
#include "tc_common.cuh"

namespace zk {

thread_local std::string g_last_error;
std::atomic<int64_t> g_launches{0};
std::atomic<int> g_fast_math{1};
std::atomic<int> g_fused{1};

zk_status fail(zk_status code, const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_last_error = buf;
    return code;
}

int sm_count() {
    static int cached[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
    if (cached[dev] == 0) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        cached[dev] = n;
    }
    return cached[dev];
}

}  // namespace zk

using namespace zk;
namespace zkapi {}
using namespace zkapi;

extern "C" {

int zk_version(void) { return 100; }
const char* zk_last_error(void) { return g_last_error.c_str(); }
int64_t zk_launch_count(void) { return g_launches.load(); }
int zk_set_fast_math(int on) { return g_fast_math.exchange(on ? 1 : 0); }
int zk_set_fused_layers(int on) { return g_fused.exchange(on ? 1 : 0); }
int zk_set_wide_min_hidden(int h) { return g_wide_min_h.exchange(h); }
int zk_set_dual_tiles(int on) { return g_dual.exchange(on ? 1 : 0); }
static thread_local cudaStream_t g_pack_stream = nullptr;
void zk_debug_timeline(long long* device_buffer) { zk::g_timeline = device_buffer; }
int zk_debug_wide_schedule(int n_linear, const int* dims, const uint8_t* const* masks_host, int univariate, int bins,
                           int features, int context, uint32_t* out_items, int max_items, uint32_t* out_rd_mask,
                           int* out_perm) {
    return zk::pair_schedule_host(1, n_linear, dims, masks_host, univariate, bins, features, context, out_items, max_items,
                                  out_rd_mask, out_perm);
}
int zk_debug_dual_schedule(int n_linear, const int* dims, const uint8_t* const* masks_host, int univariate, int bins,
                           int features, int context, uint32_t* out_items, int max_items, uint32_t* out_rd_mask,
                           int* out_perm) {
    return zk::pair_schedule_host(2, n_linear, dims, masks_host, univariate, bins, features, context, out_items, max_items,
                                  out_rd_mask, out_perm);
}
int zk_debug_watchdog_read(uint32_t* out, int n_words) {
    if (!zk::g_watch_host || !out || n_words <= 0) return 0;
    const int n = n_words < zk::W_WATCH_WORDS ? n_words : zk::W_WATCH_WORDS;
    for (int i = 0; i < n; ++i) out[i] = ((volatile uint32_t*)zk::g_watch_host)[i];
    return n;
}

zk_status zk_device_info(int* sm, int* major, int* minor) {
    int dev = 0;
    ZK_CUDA(cudaGetDevice(&dev));
    cudaDeviceProp p;
    ZK_CUDA(cudaGetDeviceProperties(&p, dev));
    if (sm) *sm = p.multiProcessorCount;
    if (major) *major = p.major;
    if (minor) *minor = p.minor;
    return ZK_OK;
}

// ---------------------------------------------------------------------------
// stand-alone bijectors
// ---------------------------------------------------------------------------
zk_status zk_rqs_forward(const float* x, int64_t ldx, const float* phi, int64_t phi_ld, int64_t B,
                         int D, int K, float bound, float slope, float* y, int64_t ldy, float* ladj,
                         int accumulate, zk_stream stream) {
    UniArgs a;
    a.univariate = ZK_UNI_RQS; a.x = x; a.ldx = ldx; a.phi = phi; a.phi_ld = phi_ld; a.B = B; a.D = D;
    a.K = K; a.bound = bound; a.slope = slope; a.y = y; a.ldy = ldy; a.ladj = ladj;
    a.accumulate = accumulate;
    a.fast_math = g_fast_math.load() != 0;
    return launch_univariate(a, (cudaStream_t)stream);
}

zk_status zk_rqs_inverse(const float* y, int64_t ldy, const float* phi, int64_t phi_ld, int64_t B,
                         int D, int K, float bound, float slope, float* x, int64_t ldx,
                         zk_stream stream) {
    UniArgs a;
    a.univariate = ZK_UNI_RQS; a.inverse = true; a.x = y; a.ldx = ldy; a.phi = phi; a.phi_ld = phi_ld;
    a.B = B; a.D = D; a.K = K; a.bound = bound; a.slope = slope; a.y = x; a.ldy = ldx;
    a.fast_math = g_fast_math.load() != 0;
    return launch_univariate(a, (cudaStream_t)stream);
}

zk_status zk_affine_forward(const float* x, int64_t ldx, const float* phi, int64_t phi_ld, int64_t B,
                            int D, float slope, float* y, int64_t ldy, float* ladj, int accumulate,
                            zk_stream stream) {
    UniArgs a;
    a.univariate = ZK_UNI_AFFINE; a.x = x; a.ldx = ldx; a.phi = phi; a.phi_ld = phi_ld; a.B = B;
    a.D = D; a.slope = slope; a.y = y; a.ldy = ldy; a.ladj = ladj; a.accumulate = accumulate;
    a.fast_math = g_fast_math.load() != 0;
    return launch_univariate(a, (cudaStream_t)stream);
}

zk_status zk_affine_inverse(const float* y, int64_t ldy, const float* phi, int64_t phi_ld, int64_t B,
                            int D, float slope, float* x, int64_t ldx, zk_stream stream) {
    UniArgs a;
    a.univariate = ZK_UNI_AFFINE; a.inverse = true; a.x = y; a.ldx = ldy; a.phi = phi;
    a.phi_ld = phi_ld; a.B = B; a.D = D; a.slope = slope; a.y = x; a.ldy = ldx;
    a.fast_math = g_fast_math.load() != 0;
    return launch_univariate(a, (cudaStream_t)stream);
}

zk_status zk_softclip_forward(const float* x, int64_t ldx, int64_t B, int D, float bound, float* y,
                              int64_t ldy, float* ladj, int accumulate, zk_stream stream) {
    return launch_softclip(x, ldx, B, D, bound, false, y, ldy, ladj, accumulate, (cudaStream_t)stream);
}
zk_status zk_softclip_inverse(const float* y, int64_t ldy, int64_t B, int D, float bound, float* x,
                              int64_t ldx, zk_stream stream) {
    return launch_softclip(y, ldy, B, D, bound, true, x, ldx, nullptr, 0, (cudaStream_t)stream);
}
zk_status zk_permute(const float* x, int64_t ldx, const int64_t* order, int64_t B, int D, float* y,
                     int64_t ldy, zk_stream stream) {
    return launch_permute(x, ldx, order, B, D, y, ldy, (cudaStream_t)stream);
}
zk_status zk_rotate(const float* x, int64_t ldx, const float* R, int transpose, int64_t B, int D,
                    float* y, int64_t ldy, zk_stream stream) {
    return launch_rotate(x, ldx, R, transpose, B, D, y, ldy, (cudaStream_t)stream);
}
zk_status zk_circular_shift(const float* x, int64_t ldx, int64_t B, int D, float bound, float* y, int64_t ldy,
                            zk_stream stream) {
    return launch_circular_shift(x, ldx, B, D, bound, y, ldy, (cudaStream_t)stream);
}
zk_status zk_box_uniform_log_prob(const float* z, int64_t ldz, const float* lower, const float* upper,
                                  const float* ladj, int64_t B, int D, float* out, zk_stream stream) {
    return launch_box_uniform(z, ldz, lower, upper, ladj, B, D, out, (cudaStream_t)stream);
}
zk_status zk_diag_normal_log_prob(const float* z, int64_t ldz, const float* loc, const float* scale,
                                  const float* ladj, int64_t B, int D, float* out, zk_stream stream) {
    return launch_diag_normal(z, ldz, loc, scale, ladj, B, D, out, (cudaStream_t)stream);
}

// ---------------------------------------------------------------------------
// conditioner handle
// ---------------------------------------------------------------------------
zk_status zk_mlp_destroy(zk_mlp* m) {
    if (!m) return ZK_OK;
    for (float* p : m->w) cudaFree(p);
    for (float* p : m->b) cudaFree(p);
    for (uint8_t* p : m->mask) cudaFree(p);
    for (float* p : m->wt) cudaFree(p);
    tc_destroy(m);
    delete m;
    return ZK_OK;
}

zk_status zk_mlp_create(const zk_mlp_desc* d, zk_mlp** out) {
    ZK_REQUIRE(d && out, "mlp_create: null argument");
    *out = nullptr;
    // the pack kernels run on the legacy default stream; the tensors they read may still be written by
    // work queued on the caller's (non-blocking) stream — zk_set_pack_stream names it
    if (g_pack_stream != nullptr) ZK_CUDA(cudaStreamSynchronize(g_pack_stream));
    ZK_REQUIRE(d->n_linear >= 1 && d->n_linear <= 64, "mlp_create: n_linear=%d out of range", d->n_linear);
    ZK_REQUIRE(d->dims && d->weight, "mlp_create: null dims/weight");
    ZK_REQUIRE(d->gemm_mode >= ZK_GEMM_AUTO && d->gemm_mode <= ZK_GEMM_BF16X1,
               "mlp_create: unknown gemm_mode %d", d->gemm_mode);
    ZK_REQUIRE(d->activation >= 0 && d->activation <= ZK_ACT_SIGMOID, "mlp_create: unknown activation %d", d->activation);
    int cnt = 0;
    ZK_CUDA(cudaGetDeviceCount(&cnt));
    zk_mlp* m = new (std::nothrow) zk_mlp();
    if (!m) return fail(ZK_ENOMEM, "mlp_create: out of host memory");
    m->n_linear = d->n_linear;
    m->act = (d->activation <= 1) ? 1 : d->activation;
    m->lact.assign(d->n_linear, m->act);
    m->lact[d->n_linear - 1] = 0;
    m->lres.assign(d->n_linear, 0);
    if (d->layer_act || d->layer_res) {  // residual conditioner: explicit per-layer pattern
        m->plain = false;
        for (int i = 0; i < d->n_linear; ++i) {
            if (d->layer_act) m->lact[i] = d->layer_act[i];
            if (d->layer_res) m->lres[i] = d->layer_res[i] ? 1 : 0;
        }
    }
    m->dims.assign(d->dims, d->dims + d->n_linear + 1);
    zk_status st = ZK_OK;
    for (int i = 0; i <= d->n_linear && st == ZK_OK; ++i)
        if (m->dims[i] <= 0) st = fail(ZK_EINVAL, "mlp_create: dims[%d]=%d", i, m->dims[i]);
    for (int i = 0; i < d->n_linear && st == ZK_OK; ++i) {
        if (m->lact[i] < 0 || m->lact[i] > ZK_ACT_SIGMOID) st = fail(ZK_EINVAL, "mlp_create: layer_act[%d]=%d", i, m->lact[i]);
        if (m->lres[i] && (i < 2 || i == d->n_linear - 1 || m->dims[i + 1] != m->dims[i - 1] || m->lact[i] != 0))
            st = fail(ZK_EINVAL, "mlp_create: layer %d cannot close a residual block (needs i >= 2, a hidden layer, equal widths, no activation)", i);
    }
    for (int i = 0; i < d->n_linear && st == ZK_OK; ++i) {
        const int64_t n = (int64_t)m->dims[i + 1] * m->dims[i];
        float *w = nullptr, *b = nullptr;
        if (!d->weight[i]) { st = fail(ZK_EINVAL, "mlp_create: weight[%d] is null", i); break; }
        if (cudaMalloc((void**)&w, n * 4) != cudaSuccess || cudaMalloc((void**)&b, ((size_t)m->dims[i + 1] + 4) * 4) != cudaSuccess /* +4: vector loads may touch one pad element */) {
            cudaFree(w);
            st = fail(ZK_ENOMEM, "mlp_create: cudaMalloc failed");
            break;
        }
        m->w.push_back(w);
        m->b.push_back(b);
        const uint8_t* mk = (d->mask ? d->mask[i] : nullptr);
        st = launch_apply_mask(d->weight[i], mk, n, w, 0);
        if (st != ZK_OK) break;
        uint8_t* mcopy = nullptr;  // kept for the backward pass: dL/dW = mask * dL/d(mask * W)
        if (mk) {
            if (cudaMalloc((void**)&mcopy, (size_t)n) != cudaSuccess) { st = fail(ZK_ENOMEM, "mlp_create: cudaMalloc failed"); break; }
            m->mask.push_back(mcopy);
            if (cudaMemcpyAsync(mcopy, mk, (size_t)n, cudaMemcpyDeviceToDevice, 0) != cudaSuccess) { st = fail(ZK_ECUDA, "mlp_create: mask copy failed"); break; }
        } else {
            m->mask.push_back(nullptr);
        }
        if (cudaMemsetAsync(b, 0, ((size_t)m->dims[i + 1] + 4) * 4, 0) != cudaSuccess) st = fail(ZK_ECUDA, "mlp_create: bias memset failed");
        if (d->bias && d->bias[i]) {
            if (cudaMemcpyAsync(b, d->bias[i], (size_t)m->dims[i + 1] * 4, cudaMemcpyDeviceToDevice, 0) != cudaSuccess)
                st = fail(ZK_ECUDA, "mlp_create: bias copy failed");
        }
        if (i < d->n_linear - 1) m->max_hidden = std::max(m->max_hidden, m->dims[i + 1]);
    }
    if (st == ZK_OK) {
        st = tc_pack(m, d->gemm_mode);  // resolves m->gemm_mode (residual blocks: per-layer GEMM kernels, never the fused ones)
    }
    if (st == ZK_OK && cudaStreamSynchronize(0) != cudaSuccess) st = fail(ZK_ECUDA, "mlp_create: sync failed");
    if (st != ZK_OK) {
        std::string keep = g_last_error;
        zk_mlp_destroy(m);
        g_last_error = keep;
        return st;
    }
    *out = m;
    return ZK_OK;
}

int zk_mlp_gemm_mode(const zk_mlp* m) { return m ? m->gemm_mode : -1; }

size_t zk_mlp_workspace_bytes(const zk_mlp* m, int64_t B) {
    if (!m || B <= 0) return 0;
    if (m->gemm_mode != ZK_GEMM_FP32) return tc_workspace_bytes(m, B);
    if (m->n_linear == 1) return 0;
    return 2 * a256((size_t)B * m->max_hidden * 4);
}

zk_status zk_mlp_forward(const zk_mlp* m, const float* x, int64_t ldx, int dx, const float* c,
                         int64_t ldc, int dc, int64_t B, float* out, int64_t ldo, void* ws,
                         size_t ws_bytes, zk_stream stream) {
    ZK_REQUIRE(m && out, "mlp_forward: null argument");
    ZK_REQUIRE(dx >= 0 && dc >= 0 && dx + dc == m->dims[0], "mlp_forward: dx(%d)+dc(%d) != in_features(%d)", dx, dc, m->dims[0]);
    ZK_REQUIRE(dx == 0 || x, "mlp_forward: null x");
    ZK_REQUIRE(dc == 0 || c, "mlp_forward: null context");
    ZK_REQUIRE(ldo >= m->dims[m->n_linear], "mlp_forward: ldo too small");
    if (B == 0) return ZK_OK;
    ZK_REQUIRE(ws_bytes >= zk_mlp_workspace_bytes(m, B), "mlp_forward: workspace too small (%zu < %zu)",
               ws_bytes, zk_mlp_workspace_bytes(m, B));
    cudaStream_t st = (cudaStream_t)stream;
    if (m->gemm_mode != ZK_GEMM_FP32)
        return tc_forward(m, x, ldx, dx, c, ldc, dc, B, out, ldo, ws, ws_bytes, st);
    Arena ar(ws, ws_bytes);
    float* h[2] = {nullptr, nullptr};
    if (m->n_linear > 1) {
        h[0] = ar.take<float>((size_t)B * m->max_hidden);
        h[1] = ar.take<float>((size_t)B * m->max_hidden);
    }
    for (int i = 0; i < m->n_linear; ++i) {
        const bool last = (i == m->n_linear - 1);
        float* dst = last ? out : h[i & 1];
        const int64_t ldd = last ? ldo : m->dims[i + 1];
        if (i == 0) {
            ZK_TRY(launch_linear_fp32(x, ldx, dx, c, ldc, m->dims[0], m->w[0], m->b[0], B, m->dims[1],
                                      m->lact[0], dst, ldd, st));
        } else {
            const float* src = h[(i - 1) & 1];
            // residual block: the input of layer i-1 lives in the buffer this layer writes (ping-pong):
            // the epilogue adds it in place
            const float* res = m->lres[i] ? dst : nullptr;
            ZK_TRY(launch_linear_fp32(src, m->dims[i], m->dims[i], nullptr, 0, m->dims[i], m->w[i],
                                      m->b[i], B, m->dims[i + 1], m->lact[i], dst, ldd, st, res, ldd));
        }
    }
    return ZK_OK;
}

// ---------------------------------------------------------------------------
// layer handle
// ---------------------------------------------------------------------------
zk_status zk_layer_destroy(zk_layer* l) {
    if (!l) return ZK_OK;
    zk_mlp_destroy(l->hyper);
    ar_inverse_free(l->inv);
    cudaFree(l->phi_shared);
    cudaFree(l->rotation);
    cudaFree(l->perm);
    cudaFree(l->perm_inv);
    cudaFree(l->idx_a);
    cudaFree(l->idx_b);
    delete l;
    return ZK_OK;
}

static zk_status layer_create_impl(const zk_layer_desc* d, zk_layer* l) {
    l->kind = d->kind; l->D = d->features; l->C = d->context; l->uni = d->univariate;
    if (l->uni == ZK_UNI_CRQS) {  // circular spline = shift + RQS over [-bound, bound] (flows/spline.py:65-72)
        l->uni = ZK_UNI_RQS;
        l->circ = true;
    }
    l->K = d->bins; l->bound = d->bound; l->slope = d->slope; l->passes = d->passes;
    ZK_REQUIRE(l->D >= 1, "layer_create: features=%d", l->D);
    ZK_REQUIRE(l->C >= 0, "layer_create: context=%d", l->C);
    const bool has_uni = (l->kind == ZK_LAYER_AUTOREGRESSIVE || l->kind == ZK_LAYER_COUPLING ||
                          l->kind == ZK_LAYER_ELEMENTWISE);
    if (has_uni) {
        ZK_REQUIRE(l->uni == ZK_UNI_AFFINE || l->uni == ZK_UNI_RQS, "layer_create: univariate=%d", d->univariate);
        if (l->uni == ZK_UNI_RQS) ZK_REQUIRE(l->K >= 1 && l->K <= 1024, "layer_create: bins=%d", l->K);
        ZK_REQUIRE(l->slope > 0.f && l->slope < 1.f, "layer_create: slope=%g", (double)l->slope);
        l->P = (l->uni == ZK_UNI_RQS) ? 3 * l->K - 1 : 2;
    }
    switch (l->kind) {
        case ZK_LAYER_AUTOREGRESSIVE: {
            ZK_REQUIRE(d->hyper, "layer_create: autoregressive layer needs a conditioner");
            ZK_REQUIRE(l->passes >= 1, "layer_create: passes=%d", l->passes);
            ZK_TRY(zk_mlp_create(d->hyper, &l->hyper));
            ZK_REQUIRE(l->hyper->dims[0] == l->D + l->C, "layer_create: conditioner in_features %d != D+C %d",
                       l->hyper->dims[0], l->D + l->C);
            ZK_REQUIRE(l->hyper->dims[l->hyper->n_linear] == l->D * l->P,
                       "layer_create: conditioner out_features %d != D*P %d",
                       l->hyper->dims[l->hyper->n_linear], l->D * l->P);
            ZK_TRY(fused_layer_prepare(l->hyper, d->hyper->mask, l->uni, l->K, l->D, l->C));
            if (d->order) l->order.assign(d->order, d->order + l->D);
            {
                int T = 0;
                size_t smem = 0;
                ZK_TRY(ar_inverse_pack(l->hyper, d->hyper->mask, d->order, l->D, l->C, l->uni, l->K, l->passes, &l->inv));
                if (l->inv && !ar_inverse_threads(l->inv, &T, &smem)) {  // state too large: use the sweeps
                    ar_inverse_free(l->inv);
                    l->inv = nullptr;
                }
            }
            return ZK_OK;
        }
        case ZK_LAYER_COUPLING: {
            ZK_REQUIRE(d->hyper && d->coupling_mask, "layer_create: coupling layer needs conditioner and mask");
            std::vector<int> ia, ib;
            for (int i = 0; i < l->D; ++i) (d->coupling_mask[i] ? ia : ib).push_back(i);
            l->n_a = (int)ia.size();
            l->n_b = (int)ib.size();
            ZK_REQUIRE(l->n_a > 0 && l->n_b > 0, "layer_create: coupling mask must split the features");
            ZK_TRY(dev_copy_from_host(ia.data(), ia.size(), &l->idx_a));
            ZK_TRY(dev_copy_from_host(ib.data(), ib.size(), &l->idx_b));
            ZK_TRY(zk_mlp_create(d->hyper, &l->hyper));
            ZK_REQUIRE(l->hyper->dims[0] == l->n_a + l->C, "layer_create: coupling conditioner in_features mismatch");
            ZK_REQUIRE(l->hyper->dims[l->hyper->n_linear] == l->n_b * l->P, "layer_create: coupling conditioner out_features mismatch");
            return ZK_OK;
        }
        case ZK_LAYER_ELEMENTWISE: {
            if (d->hyper) {
                ZK_REQUIRE(l->C > 0, "layer_create: elementwise conditioner needs context");
                ZK_TRY(zk_mlp_create(d->hyper, &l->hyper));
                ZK_REQUIRE(l->hyper->dims[0] == l->C && l->hyper->dims[l->hyper->n_linear] == l->D * l->P,
                           "layer_create: elementwise conditioner shape mismatch");
            } else {
                ZK_REQUIRE(d->phi, "layer_create: elementwise layer needs phi or a conditioner");
                ZK_CUDA(cudaMalloc((void**)&l->phi_shared, (size_t)l->D * l->P * 4));
                ZK_CUDA(cudaMemcpy(l->phi_shared, d->phi, (size_t)l->D * l->P * 4, cudaMemcpyDeviceToDevice));
            }
            return ZK_OK;
        }
        case ZK_LAYER_SOFTCLIP:
            ZK_REQUIRE(l->bound > 0.f, "layer_create: softclip bound=%g", (double)l->bound);
            return ZK_OK;
        case ZK_LAYER_PERMUTATION: {
            ZK_REQUIRE(d->order, "layer_create: permutation needs order");
            std::vector<int64_t> ord(d->order, d->order + l->D), inv(l->D, -1);
            for (int i = 0; i < l->D; ++i) {
                ZK_REQUIRE(ord[i] >= 0 && ord[i] < l->D && inv[ord[i]] < 0, "layer_create: order is not a permutation");
                inv[ord[i]] = i;  // argsort(order), transforms.py:1210-1211
            }
            ZK_TRY(dev_copy_from_host(ord.data(), ord.size(), &l->perm));
            ZK_TRY(dev_copy_from_host(inv.data(), inv.size(), &l->perm_inv));
            return ZK_OK;
        }
        case ZK_LAYER_ROTATION: {
            ZK_REQUIRE(d->rotation, "layer_create: rotation needs R");
            ZK_CUDA(cudaMalloc((void**)&l->rotation, (size_t)l->D * l->D * 4));
            ZK_CUDA(cudaMemcpy(l->rotation, d->rotation, (size_t)l->D * l->D * 4, cudaMemcpyDeviceToDevice));
            return ZK_OK;
        }
        default:
            return fail(ZK_EUNSUPPORTED, "layer_create: unknown layer kind %d", d->kind);
    }
}

zk_status zk_layer_create(const zk_layer_desc* d, zk_layer** out) {
    ZK_REQUIRE(d && out, "layer_create: null argument");
    *out = nullptr;
    int cnt = 0;
    ZK_CUDA(cudaGetDeviceCount(&cnt));
    zk_layer* l = new (std::nothrow) zk_layer();
    if (!l) return fail(ZK_ENOMEM, "layer_create: out of host memory");
    zk_status st = layer_create_impl(d, l);
    if (st != ZK_OK) {
        std::string keep = g_last_error;
        zk_layer_destroy(l);
        g_last_error = keep;
        return st;
    }
    *out = l;
    return ZK_OK;
}

void zk_set_pack_stream(zk_stream stream) { g_pack_stream = (cudaStream_t)stream; }

zk_status zk_layer_update_weights(zk_layer* l, const float* const* weight, const float* const* bias, zk_stream stream) {
    ZK_REQUIRE(l && weight, "layer_update_weights: null argument");
    ZK_REQUIRE(l->hyper, "layer_update_weights: the layer has no conditioner");
    zk_mlp* m = l->hyper;
    cudaStream_t st = (cudaStream_t)stream;
    for (int i = 0; i < m->n_linear; ++i) {
        ZK_REQUIRE(weight[i], "layer_update_weights: weight[%d] is null", i);
        const int64_t n = (int64_t)m->dims[i + 1] * m->dims[i];
        ZK_TRY(launch_apply_mask(weight[i], m->mask[i], n, m->w[i], st));  // nn.py:218 `mask * W`, once per update
        if (bias && bias[i]) ZK_CUDA(cudaMemcpyAsync(m->b[i], bias[i], (size_t)m->dims[i + 1] * 4, cudaMemcpyDeviceToDevice, st));
    }
    ZK_TRY(tc_refresh(m, st));
    ZK_TRY(fused_refresh(m, st));
    m->bwd_dirty = true;          // transposed weights / backward planes: refilled by the next backward call
    if (l->inv) l->inv_dirty = true;  // step-ordered inverse stream: rebuilt by the next inverse call
    return ZK_OK;
}

int zk_layer_sequential_inverse(const zk_layer* l) {
    return (l && l->kind == ZK_LAYER_AUTOREGRESSIVE && (l->inv != nullptr || l->inv_dirty)) ? 1 : 0;
}

int zk_layer_fused_info(const zk_layer* l, double* out) {
    if (!l || !out) return -1;
    out[0] = out[1] = out[2] = out[3] = 0.0;
    if (l->kind != ZK_LAYER_AUTOREGRESSIVE || !l->hyper) return 0;
    const zk_mlp* m = l->hyper;
    double dense = 0;
    for (int i = 0; i < m->n_linear; ++i) dense += (double)m->dims[i] * m->dims[i + 1];
    out[3] = dense;
    const TcPack* pk = tc_pack_of(m);
    if (!pk || l->circ || !fused_layer_supported(m, l->uni, l->K, l->D, l->C)) return 0;
    const int kind = fused_layer_kind(m, l->uni, l->K, l->D, l->C);
    out[0] = kind;
    if (kind == 1) {
        out[1] = pk->fused.n_items;
        out[2] = pk->fused.issued_macs_per_row;
    } else {
        const WidePack& wp = (kind == 3) ? pk->dual : pk->wide;
        out[1] = wp.n_items;
        out[2] = wp.issued_macs_per_row;
    }
    return kind;
}

size_t zk_layer_workspace_bytes(const zk_layer* l, int64_t B) {
    if (!l || B <= 0) return 0;
    switch (l->kind) {
        case ZK_LAYER_AUTOREGRESSIVE:
            return a256((size_t)B * l->D * l->P * 4) + zk_mlp_workspace_bytes(l->hyper, B);
        case ZK_LAYER_COUPLING:
            return a256((size_t)B * l->n_b * l->P * 4) + a256((size_t)B * l->n_a * 4) +
                   zk_mlp_workspace_bytes(l->hyper, B);
        case ZK_LAYER_ELEMENTWISE:
            return l->hyper ? a256((size_t)B * l->D * l->P * 4) + zk_mlp_workspace_bytes(l->hyper, B) : 0;
        default:
            return 0;
    }
}

}  // extern "C"

namespace zkapi {

// gather of the constant split: xa[:, j] = x[:, idx_a[j]] (transforms.py:1040-1041)
__global__ void gather_columns_kernel(const float* x, int64_t ldx, const int* cols, int n, int64_t B,
                                      float* out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * n) return;
    const int64_t r = i / n;
    const int j = (int)(i - r * n);
    out[r * n + j] = x[r * ldx + cols[j]];
}

__global__ void copy_rows_kernel(const float* x, int64_t ldx, int64_t B, int D, float* y, int64_t ldy) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * D) return;
    const int64_t r = i / D;
    const int d = (int)(i - r * D);
    y[r * ldy + d] = x[r * ldx + d];
}

zk_status copy_rows(const float* x, int64_t ldx, int64_t B, int D, float* y, int64_t ldy, cudaStream_t st) {
    if (B == 0) return ZK_OK;
    copy_rows_kernel<<<(unsigned)ceil_div(B * D, 256), 256, 0, st>>>(x, ldx, B, D, y, ldy);
    return check_launch("copy_rows_kernel");
}

bool layer_can_fuse_base(const zk_layer* l) {
    return l->kind == ZK_LAYER_AUTOREGRESSIVE || l->kind == ZK_LAYER_ELEMENTWISE;
}

// Forward of one layer.  When log_prob != nullptr (only for layers where
// layer_can_fuse_base) the DiagNormal term is fused and y may be nullptr.
zk_status layer_forward_impl(const zk_layer* l, const float* x, int64_t ldx, const float* c,
                             int64_t ldc, int64_t B, float* y, int64_t ldy, float* ladj,
                             int accumulate, float* log_prob, const float* loc, const float* scale,
                             void* ws, size_t ws_bytes, cudaStream_t st) {
    if (B == 0) return ZK_OK;
    ZK_REQUIRE(l->C == 0 || c != nullptr, "layer needs a context of %d features", l->C);
    Arena ar(ws, ws_bytes);
    UniArgs a;
    a.univariate = l->uni; a.B = B; a.K = l->K; a.bound = l->bound; a.slope = l->slope;
    a.ladj = ladj; a.accumulate = accumulate; a.log_prob = log_prob; a.base_loc = loc;
    a.base_scale = scale; a.fast_math = g_fast_math.load() != 0; a.circular = l->circ;
    switch (l->kind) {
        case ZK_LAYER_AUTOREGRESSIVE: {
            // transforms.py:1005-1007 + flows/autoregressive.py:207-215
            if (g_fused.load() && !l->circ && fused_layer_supported(l->hyper, l->uni, l->K, l->D, l->C)) {
                // ONE kernel: conditioner GEMMs + bijector + ladj; neither the hidden
                // activations nor phi touch HBM
                FusedLayerArgs f;
                f.univariate = l->uni; f.bins = l->K; f.D = l->D; f.C = l->C; f.bound = l->bound;
                f.slope = l->slope; f.x = x; f.ldx = ldx; f.c = c; f.ldc = ldc; f.B = B; f.y = y; f.ldy = ldy;
                f.ladj = ladj; f.accumulate = accumulate; f.log_prob = log_prob; f.base_loc = loc;
                f.base_scale = scale; f.fast_math = g_fast_math.load() != 0;
                return launch_fused_layer(l->hyper, f, st);
            }
            float* phi = ar.take<float>((size_t)B * l->D * l->P);
            ZK_REQUIRE(ar.ok, "layer_forward: workspace too small");
            ZK_TRY(zk_mlp_forward(l->hyper, x, ldx, l->D, c, ldc, l->C, B, phi, (int64_t)l->D * l->P,
                                  ar.base + ar.off, ar.size - ar.off, st));
            a.x = x; a.ldx = ldx; a.phi = phi; a.phi_ld = (int64_t)l->D * l->P; a.D = l->D;
            a.y = y; a.ldy = ldy;
            return launch_univariate(a, st);
        }
        case ZK_LAYER_COUPLING: {
            // transforms.py:1067-1072 + flows/coupling.py:128-136
            float* phi = ar.take<float>((size_t)B * l->n_b * l->P);
            float* xa = ar.take<float>((size_t)B * l->n_a);
            ZK_REQUIRE(ar.ok, "layer_forward: workspace too small");
            gather_columns_kernel<<<(unsigned)ceil_div(B * l->n_a, 256), 256, 0, st>>>(x, ldx, l->idx_a, l->n_a, B, xa);
            ZK_TRY(check_launch("gather_columns_kernel"));
            ZK_TRY(zk_mlp_forward(l->hyper, xa, l->n_a, l->n_a, c, ldc, l->C, B, phi, (int64_t)l->n_b * l->P,
                                  ar.base + ar.off, ar.size - ar.off, st));
            if (y) ZK_TRY(launch_copy_columns(x, ldx, l->idx_a, l->n_a, B, y, ldy, st));
            a.x = x; a.ldx = ldx; a.phi = phi; a.phi_ld = (int64_t)l->n_b * l->P; a.D = l->n_b;
            a.y = y; a.ldy = ldy; a.dim_map = l->idx_b;
            return launch_univariate(a, st);
        }
        case ZK_LAYER_ELEMENTWISE: {
            // flows/gaussianization.py:86-94
            a.x = x; a.ldx = ldx; a.D = l->D; a.y = y; a.ldy = ldy;
            if (l->hyper) {
                const int64_t rows = (ldc == 0) ? 1 : B;  // broadcast context => one shared table
                float* phi = ar.take<float>((size_t)rows * l->D * l->P);
                ZK_REQUIRE(ar.ok, "layer_forward: workspace too small");
                ZK_TRY(zk_mlp_forward(l->hyper, c, ldc, l->C, nullptr, 0, 0, rows, phi, (int64_t)l->D * l->P,
                                      ar.base + ar.off, ar.size - ar.off, st));
                a.phi = phi;
                a.phi_ld = (ldc == 0) ? 0 : (int64_t)l->D * l->P;
            } else {
                a.phi = l->phi_shared;
                a.phi_ld = 0;
            }
            return launch_univariate(a, st);
        }
        case ZK_LAYER_SOFTCLIP:
            return launch_softclip(x, ldx, B, l->D, l->bound, false, y, ldy, ladj, accumulate, st);
        case ZK_LAYER_PERMUTATION:
            ZK_TRY(launch_permute(x, ldx, l->perm, B, l->D, y, ldy, st));
            if (ladj && !accumulate) ZK_TRY(launch_fill(ladj, B, 0.f, st));  // transforms.py:1213-1214
            return ZK_OK;
        case ZK_LAYER_ROTATION:
            ZK_TRY(launch_rotate(x, ldx, l->rotation, 0, B, l->D, y, ldy, st));
            if (ladj && !accumulate) ZK_TRY(launch_fill(ladj, B, 0.f, st));  // transforms.py:1243-1244
            return ZK_OK;
    }
    return fail(ZK_EUNSUPPORTED, "layer_forward: unknown kind %d", l->kind);
}

// Inverse of one layer.  With `ladj` the layer ALSO adds (accumulate) / writes the per-sample FORWARD
// log-determinant at the solution — and with `base_lp` the base log-density of its input y — when its
// inverse kernel can produce them in the same sweep; *ladj_done tells the caller whether it did
// (otherwise the caller evaluates the layer's forward ladj separately).
zk_status layer_inverse_impl(const zk_layer* l, const float* y, int64_t ldy, const float* c,
                             int64_t ldc, int64_t B, float* x, int64_t ldx, void* ws,
                             size_t ws_bytes, cudaStream_t st, float* ladj, int accumulate, bool base_lp,
                             const float* base_loc, const float* base_scale, bool* ladj_done, bool as_member = false) {
    if (ladj_done) *ladj_done = false;
    if (B == 0) return ZK_OK;
    ZK_REQUIRE(l->C == 0 || c != nullptr, "layer needs a context of %d features", l->C);
    Arena ar(ws, ws_bytes);
    UniArgs a;
    a.univariate = l->uni; a.inverse = true; a.B = B; a.K = l->K; a.bound = l->bound;
    a.slope = l->slope; a.fast_math = g_fast_math.load() != 0; a.circular = l->circ;
    switch (l->kind) {
        case ZK_LAYER_AUTOREGRESSIVE: {
            // transforms.py:994-1000: x = zeros_like(y); for _ in range(passes): x = meta(x).inv(y)
            if (l->inv_dirty) {  // the weights were refreshed in place: rebuild the step-ordered stream once
                static std::mutex mu;
                std::lock_guard<std::mutex> lk(mu);
                zk_layer* ml = const_cast<zk_layer*>(l);
                if (ml->inv_dirty) {
                    ZK_CUDA(cudaStreamSynchronize(st));  // the refresh kernels ran on the caller's stream
                    ar_inverse_free(ml->inv);
                    ml->inv = nullptr;
                    int T = 0;
                    size_t smem = 0;
                    ZK_TRY(ar_inverse_pack(ml->hyper, ml->hyper->mask.data(), ml->order.empty() ? nullptr : ml->order.data(), ml->D,
                                           ml->C, ml->uni, ml->K, ml->passes, &ml->inv));
                    if (ml->inv && !ar_inverse_threads(ml->inv, &T, &smem)) {
                        ar_inverse_free(ml->inv);
                        ml->inv = nullptr;
                    }
                    ml->inv_dirty = false;
                }
            }
            if (l->inv && g_fused.load()) {  // same fixed point, every weight visited once (ar_inverse.cu)
                ArInvArgs ia;
                ia.y = y; ia.ldy = ldy; ia.c = c; ia.ldc = ldc; ia.B = B; ia.x = x; ia.ldx = ldx;
                ia.bound = l->bound; ia.slope = l->slope; ia.fast = g_fast_math.load() != 0; ia.circular = l->circ;
                if (ladj) {
                    ia.ladj = ladj; ia.accumulate = accumulate; ia.base = base_lp; ia.base_loc = base_loc; ia.base_scale = base_scale;
                    ia.as_inverse_member = as_member;
                    if (ladj_done) *ladj_done = true;
                }
                return launch_ar_inverse(l->inv, ia, st);
            }
            float* phi = ar.take<float>((size_t)B * l->D * l->P);
            ZK_REQUIRE(ar.ok, "layer_inverse: workspace too small");
            if (ldx == l->D) {
                ZK_CUDA(cudaMemsetAsync(x, 0, (size_t)B * l->D * 4, st));
            } else {
                ZK_CUDA(cudaMemset2DAsync(x, (size_t)ldx * 4, 0, (size_t)l->D * 4, (size_t)B, st));
            }
            a.x = y; a.ldx = ldy; a.phi = phi; a.phi_ld = (int64_t)l->D * l->P; a.D = l->D;
            a.y = x; a.ldy = ldx;
            for (int p = 0; p < l->passes; ++p) {
                ZK_TRY(zk_mlp_forward(l->hyper, x, ldx, l->D, c, ldc, l->C, B, phi, (int64_t)l->D * l->P,
                                      ar.base + ar.off, ar.size - ar.off, st));
                ZK_TRY(launch_univariate(a, st));
            }
            return ZK_OK;
        }
        case ZK_LAYER_COUPLING: {
            // transforms.py:1054-1058
            float* phi = ar.take<float>((size_t)B * l->n_b * l->P);
            float* ya = ar.take<float>((size_t)B * l->n_a);
            ZK_REQUIRE(ar.ok, "layer_inverse: workspace too small");
            gather_columns_kernel<<<(unsigned)ceil_div(B * l->n_a, 256), 256, 0, st>>>(y, ldy, l->idx_a, l->n_a, B, ya);
            ZK_TRY(check_launch("gather_columns_kernel"));
            ZK_TRY(zk_mlp_forward(l->hyper, ya, l->n_a, l->n_a, c, ldc, l->C, B, phi, (int64_t)l->n_b * l->P,
                                  ar.base + ar.off, ar.size - ar.off, st));
            ZK_TRY(launch_copy_columns(y, ldy, l->idx_a, l->n_a, B, x, ldx, st));
            a.x = y; a.ldx = ldy; a.phi = phi; a.phi_ld = (int64_t)l->n_b * l->P; a.D = l->n_b;
            a.y = x; a.ldy = ldx; a.dim_map = l->idx_b;
            return launch_univariate(a, st);
        }
        case ZK_LAYER_ELEMENTWISE: {
            a.x = y; a.ldx = ldy; a.D = l->D; a.y = x; a.ldy = ldx;
            if (l->hyper) {
                const int64_t rows = (ldc == 0) ? 1 : B;
                float* phi = ar.take<float>((size_t)rows * l->D * l->P);
                ZK_REQUIRE(ar.ok, "layer_inverse: workspace too small");
                ZK_TRY(zk_mlp_forward(l->hyper, c, ldc, l->C, nullptr, 0, 0, rows, phi, (int64_t)l->D * l->P,
                                      ar.base + ar.off, ar.size - ar.off, st));
                a.phi = phi;
                a.phi_ld = (ldc == 0) ? 0 : (int64_t)l->D * l->P;
            } else {
                a.phi = l->phi_shared;
                a.phi_ld = 0;
            }
            return launch_univariate(a, st);
        }
        case ZK_LAYER_SOFTCLIP:
            return launch_softclip(y, ldy, B, l->D, l->bound, true, x, ldx, nullptr, 0, st);
        case ZK_LAYER_PERMUTATION:
            return launch_permute(y, ldy, l->perm_inv, B, l->D, x, ldx, st);
        case ZK_LAYER_ROTATION:
            return launch_rotate(y, ldy, l->rotation, 1, B, l->D, x, ldx, st);
    }
    return fail(ZK_EUNSUPPORTED, "layer_inverse: unknown kind %d", l->kind);
}

// ---- flow-level helpers ----
struct FlowPlan {
    size_t per_row = 0;  // bytes of workspace per batch row (upper bound incl. alignment slack)
    size_t fixed = 0;    // fixed bytes
};

// scratch one layer needs beyond its input / output for ONE direction, with the kernels that will
// actually run (a fused forward layer or a dimension-sequential inverse layer keeps phi and the hidden
// activations on chip: nothing), dir: 1 forward, 2 inverse, 0 either (the public, conservative figure)
size_t layer_ws_dir(const zk_layer* l, int64_t Bc, int dir) {
    if (dir != 0 && l->kind == ZK_LAYER_AUTOREGRESSIVE && g_fused.load()) {
        const bool fwd_fused = !l->circ && fused_layer_supported(l->hyper, l->uni, l->K, l->D, l->C);
        const bool inv_seq = (l->inv != nullptr || l->inv_dirty);
        if (dir == 1 && fwd_fused) return 0;
        if (dir == 2 && inv_seq) return 0;
    }
    return zk_layer_workspace_bytes(l, Bc);
}

size_t flow_ws_for(const zk_flow_desc* f, int64_t Bc, int dir = 0) {
    const int D = f->features;
    size_t layer_max = 0;
    for (int i = 0; i < f->n_layers; ++i) {
        size_t need = layer_ws_dir(f->layers[i], Bc, dir);
        // inverse + log_prob: a layer whose inverse kernel cannot emit its ladj runs its forward as well
        if (dir == 2 && need != 0) need = std::max(need, layer_ws_dir(f->layers[i], Bc, 1));
        layer_max = std::max(layer_max, need);
    }
    return 2 * a256((size_t)Bc * D * 4)      // ping-pong activations
           + a256((size_t)Bc * 4)            // ladj
           + a256((size_t)Bc * D * 4)        // x scratch for inverse + log_prob
           + a256(reduce_scratch_bytes()) + layer_max + 1024;
}

int64_t flow_chunk_rows(const zk_flow_desc* f, int64_t B, size_t ws_bytes, int dir = 0) {
    if (flow_ws_for(f, B, dir) <= ws_bytes) return B;
    int64_t lo = 1, hi = B;  // largest chunk that fits (monotone in Bc)
    if (flow_ws_for(f, 1, dir) > ws_bytes) return 0;
    while (lo < hi) {
        int64_t mid = lo + (hi - lo + 1) / 2;
        if (flow_ws_for(f, mid, dir) <= ws_bytes) lo = mid; else hi = mid - 1;
    }
    // keep tiles aligned: round down to a multiple of 1024 rows when possible
    if (lo >= 2048) lo = lo / 1024 * 1024;
    return lo;
}

zk_status flow_check(const zk_flow_desc* f) {
    ZK_REQUIRE(f, "flow: null descriptor");
    ZK_REQUIRE(f->n_layers >= 0 && (f->n_layers == 0 || f->layers), "flow: bad layer list");
    ZK_REQUIRE(f->features >= 1 && f->context >= 0, "flow: bad features/context");
    ZK_REQUIRE((f->base_loc == nullptr) == (f->base_scale == nullptr), "flow: base loc/scale must both be set or null");
    ZK_REQUIRE(f->base_kind == ZK_BASE_DIAG_NORMAL || f->base_kind == ZK_BASE_BOX_UNIFORM, "flow: unknown base kind %d", f->base_kind);
    ZK_REQUIRE(f->base_kind != ZK_BASE_BOX_UNIFORM || f->base_loc, "flow: a BoxUniform base needs lower / upper bounds");
    for (int i = 0; i < f->n_layers; ++i) {
        const zk_layer* l = f->layers[i];
        ZK_REQUIRE(l, "flow: layer %d is null", i);
        ZK_REQUIRE(l->D == f->features, "flow: layer %d has %d features, flow has %d", i, l->D, f->features);
        ZK_REQUIRE(l->C == 0 || l->C == f->context, "flow: layer %d expects context %d, flow has %d", i, l->C, f->context);
        if (f->inverted && f->inverted[i])
            ZK_REQUIRE(zk_layer_sequential_inverse(l), "flow: member %d is inverted but its layer has no dimension-sequential inverse", i);
    }
    return ZK_OK;
}

// forward over one chunk; mode 0: (z, ladj); mode 1: log_prob
zk_status flow_forward_chunk(const zk_flow_desc* f, const float* x, int64_t ldx, const float* c,
                             int64_t ldc, int64_t B, float* z, int64_t ldz, float* ladj_out,
                             float* log_prob, void* ws, size_t ws_bytes, cudaStream_t st) {
    const int D = f->features, T = f->n_layers;
    Arena ar(ws, ws_bytes);
    float* buf[2] = {ar.take<float>((size_t)B * D), ar.take<float>((size_t)B * D)};
    float* ladj = ladj_out ? ladj_out : ar.take<float>((size_t)B);
    ZK_REQUIRE(ar.ok, "flow: workspace too small");
    void* lws = ar.base + ar.off;
    const size_t lws_bytes = ar.size - ar.off;
    const float* cur = x;
    int64_t ldcur = ldx;
    bool fused = false;
    for (int i = 0; i < T; ++i) {
        const zk_layer* l = f->layers[i];
        const bool last = (i == T - 1);
        const float* cc = l->C ? c : nullptr;
        if (f->inverted && f->inverted[i]) {
            // LazyInverse member (lazy.py:81-98): forward of the member = the layer's dimension-sequential
            // inverse; its ladj = - ladj_layer at the solution, accumulated by the same kernel, which also adds
            // the DiagNormal density of its OUTPUT when it closes a log_prob call
            const bool fuse_base = last && log_prob && f->base_kind == ZK_BASE_DIAG_NORMAL;
            float* dst = (last && z) ? z : buf[i & 1];
            const int64_t ldd = (last && z) ? ldz : D;
            float* acc = ladj;
            if (fuse_base) {  // the closing kernel writes log_prob itself: hand it what the earlier members summed
                if (i > 0) ZK_CUDA(cudaMemcpyAsync(log_prob, ladj, (size_t)B * 4, cudaMemcpyDeviceToDevice, st));
                acc = log_prob;
            }
            bool done = false;
            ZK_TRY(layer_inverse_impl(l, cur, ldcur, cc, ldc, B, dst, ldd, lws, lws_bytes, st, acc, i > 0 ? 1 : 0,
                                      fuse_base, f->base_loc, f->base_scale, &done, true));
            ZK_REQUIRE(done, "flow: member %d is inverted but its layer has no dimension-sequential inverse", i);
            cur = dst;
            ldcur = ldd;
            if (fuse_base) {
                fused = true;
                break;
            }
            continue;
        }
        if (last && log_prob && layer_can_fuse_base(l) && f->base_kind == ZK_BASE_DIAG_NORMAL) {
            ZK_TRY(layer_forward_impl(l, cur, ldcur, cc, ldc, B, nullptr, 0, ladj, i > 0, log_prob,
                                      f->base_loc, f->base_scale, lws, lws_bytes, st));
            fused = true;
            break;
        }
        float* dst = (last && z) ? z : buf[i & 1];
        const int64_t ldd = (last && z) ? ldz : D;
        ZK_TRY(layer_forward_impl(l, cur, ldcur, cc, ldc, B, dst, ldd, ladj, i > 0, nullptr, nullptr,
                                  nullptr, lws, lws_bytes, st));
        cur = dst;
        ldcur = ldd;
    }
    if (T == 0) {
        ZK_TRY(launch_fill(ladj, B, 0.f, st));
        if (z) ZK_TRY(copy_rows(x, ldx, B, D, z, ldz, st));
    }
    if (log_prob && !fused) {
        if (f->base_kind == ZK_BASE_BOX_UNIFORM)
            ZK_TRY(launch_box_uniform(cur, ldcur, f->base_loc, f->base_scale, ladj, B, D, log_prob, st));
        else
            ZK_TRY(launch_diag_normal(cur, ldcur, f->base_loc, f->base_scale, ladj, B, D, log_prob, st));
    }
    return ZK_OK;
}

zk_status flow_inverse_chunk(const zk_flow_desc* f, const float* z, int64_t ldz, const float* c,
                             int64_t ldc, int64_t B, float* x, int64_t ldx, float* log_prob,
                             void* ws, size_t ws_bytes, cudaStream_t st) {
    const int D = f->features, T = f->n_layers;
    Arena ar(ws, ws_bytes);
    float* buf[2] = {ar.take<float>((size_t)B * D), ar.take<float>((size_t)B * D)};
    ZK_REQUIRE(ar.ok, "flow: workspace too small");
    void* lws = ar.base + ar.off;
    const size_t lws_bytes = ar.size - ar.off;
    const float* cur = z;
    int64_t ldcur = ldz;
    // distributions.py:129-138: log p(x) = base.log_prob(z) - ladj_inv, and ladj_inv = -ladj_fwd(x)
    // (torch/distributions/transforms.py:277-280).  ONE sweep: every layer's inverse kernel also
    // accumulates its forward ladj at the solution (and the first one the base log-density of z)
    // into `log_prob`; only layers whose inverse kernel cannot (sweep-based inverses, coupling,
    // element-wise tables) pay a forward evaluation of that layer alone.
    const bool want = (log_prob != nullptr);
    bool seeded = false;  // log_prob already holds the base term (+ earlier layers)
    for (int i = T - 1; i >= 0; --i) {
        const zk_layer* l = f->layers[i];
        const bool last = (i == 0);
        float* dst = last ? x : buf[i & 1];
        const int64_t ldd = last ? ldx : D;
        if (f->inverted && f->inverted[i]) {
            // inverse of a LazyInverse member = the layer's forward (its y; the ladj is not needed without log_prob)
            ZK_REQUIRE(!want, "flow_inverse: log_prob of a flow with inverted members is not fused (use log_prob(x) of the result)");
            ZK_TRY(layer_forward_impl(l, cur, ldcur, l->C ? c : nullptr, ldc, B, dst, ldd, nullptr, 0, nullptr, nullptr, nullptr,
                                      lws, lws_bytes, st));
            cur = dst;
            ldcur = ldd;
            continue;
        }
        bool done = false;
        // the DiagNormal term of z can ride in the first inverted layer's kernel; a BoxUniform base is seeded apart
        const bool can_seed = want && !seeded && i == T - 1 && f->base_kind != ZK_BASE_BOX_UNIFORM;
        if (want && !seeded && !can_seed) {
            ZK_TRY(launch_box_uniform(z, ldz, f->base_loc, f->base_scale, nullptr, B, D, log_prob, st));
            seeded = true;
        }
        ZK_TRY(layer_inverse_impl(l, cur, ldcur, l->C ? c : nullptr, ldc, B, dst, ldd, lws, lws_bytes, st,
                                  want ? log_prob : nullptr, seeded ? 1 : 0, can_seed, f->base_loc, f->base_scale, &done));
        if (want) {
            if (done) {
                seeded = true;
            } else {
                if (!seeded) {  // base log-density of z = the first inverted layer's input
                    if (f->base_kind == ZK_BASE_BOX_UNIFORM)
                        ZK_TRY(launch_box_uniform(z, ldz, f->base_loc, f->base_scale, nullptr, B, D, log_prob, st));
                    else
                        ZK_TRY(launch_diag_normal(z, ldz, f->base_loc, f->base_scale, nullptr, B, D, log_prob, st));
                    seeded = true;
                }
                // forward ladj of this layer alone at its input `dst`; its output is not needed and goes to
                // the other ping-pong buffer (it holds this layer's y, which is dead now; never the caller's z)
                float* scratch = buf[(i + 1) & 1];
                if (l->kind != ZK_LAYER_PERMUTATION && l->kind != ZK_LAYER_ROTATION)  // those have ladj = 0
                    ZK_TRY(layer_forward_impl(l, dst, ldd, l->C ? c : nullptr, ldc, B, scratch, D, log_prob, 1, nullptr,
                                              nullptr, nullptr, lws, lws_bytes, st));
            }
        }
        cur = dst;
        ldcur = ldd;
    }
    if (T == 0) {
        ZK_TRY(copy_rows(z, ldz, B, D, x, ldx, st));
        if (want) {
            if (f->base_kind == ZK_BASE_BOX_UNIFORM)
                ZK_TRY(launch_box_uniform(z, ldz, f->base_loc, f->base_scale, nullptr, B, D, log_prob, st));
            else
                ZK_TRY(launch_diag_normal(z, ldz, f->base_loc, f->base_scale, nullptr, B, D, log_prob, st));
        }
    }
    return ZK_OK;
}

}  // namespace zkapi

extern "C" {

zk_status zk_layer_forward(const zk_layer* l, const float* x, int64_t ldx, const float* c, int64_t ldc,
                           int64_t B, float* y, int64_t ldy, float* ladj, int accumulate, void* ws,
                           size_t ws_bytes, zk_stream stream) {
    ZK_REQUIRE(l && x && y, "layer_forward: null argument");
    ZK_REQUIRE(x != y, "layer_forward: y must not alias x");
    ZK_REQUIRE(B >= 0 && ldx >= l->D && ldy >= l->D, "layer_forward: bad shape");
    ZK_REQUIRE(ws_bytes >= zk_layer_workspace_bytes(l, B), "layer_forward: workspace too small");
    return layer_forward_impl(l, x, ldx, c, ldc, B, y, ldy, ladj, accumulate, nullptr, nullptr, nullptr,
                              ws, ws_bytes, (cudaStream_t)stream);
}

zk_status zk_layer_inverse(const zk_layer* l, const float* y, int64_t ldy, const float* c, int64_t ldc,
                           int64_t B, float* x, int64_t ldx, void* ws, size_t ws_bytes,
                           zk_stream stream) {
    ZK_REQUIRE(l && x && y, "layer_inverse: null argument");
    ZK_REQUIRE(x != y, "layer_inverse: x must not alias y");
    ZK_REQUIRE(B >= 0 && ldx >= l->D && ldy >= l->D, "layer_inverse: bad shape");
    ZK_REQUIRE(ws_bytes >= zk_layer_workspace_bytes(l, B), "layer_inverse: workspace too small");
    return layer_inverse_impl(l, y, ldy, c, ldc, B, x, ldx, ws, ws_bytes, (cudaStream_t)stream, nullptr, 0, false,
                              nullptr, nullptr, nullptr);
}

size_t zk_flow_workspace_bytes(const zk_flow_desc* f, int64_t B) {
    if (!f || B <= 0) return 1024;
    return flow_ws_for(f, B);
}
size_t zk_flow_min_workspace_bytes(const zk_flow_desc* f) { return f ? flow_ws_for(f, 1) : 1024; }

zk_status zk_flow_forward(const zk_flow_desc* f, const float* x, int64_t ldx, const float* c,
                          int64_t ldc, int64_t B, float* z, int64_t ldz, float* ladj, void* ws,
                          size_t ws_bytes, zk_stream stream) {
    ZK_TRY(flow_check(f));
    ZK_REQUIRE(x && z && ladj, "flow_forward: null argument");
    ZK_REQUIRE(x != z, "flow_forward: z must not alias x");
    ZK_REQUIRE(B >= 0 && ldx >= f->features && ldz >= f->features, "flow_forward: bad shape");
    ZK_REQUIRE(f->context == 0 || c, "flow_forward: flow needs a context");
    if (B == 0) return ZK_OK;
    const int64_t Bc = flow_chunk_rows(f, B, ws_bytes, 1);
    ZK_REQUIRE(Bc > 0, "flow_forward: workspace too small (%zu < %zu)", ws_bytes, zk_flow_min_workspace_bytes(f));
    for (int64_t i0 = 0; i0 < B; i0 += Bc) {
        const int64_t n = std::min(Bc, B - i0);
        ZK_TRY(flow_forward_chunk(f, x + i0 * ldx, ldx, c ? c + i0 * ldc : nullptr, ldc, n, z + i0 * ldz,
                                  ldz, ladj + i0, nullptr, ws, ws_bytes, (cudaStream_t)stream));
    }
    return ZK_OK;
}

zk_status zk_flow_log_prob(const zk_flow_desc* f, const float* x, int64_t ldx, const float* c,
                           int64_t ldc, int64_t B, float* log_prob, double* sum_log_prob, void* ws,
                           size_t ws_bytes, zk_stream stream) {
    ZK_TRY(flow_check(f));
    ZK_REQUIRE(x && log_prob, "flow_log_prob: null argument");
    ZK_REQUIRE(B >= 0 && ldx >= f->features, "flow_log_prob: bad shape");
    ZK_REQUIRE(f->context == 0 || c, "flow_log_prob: flow needs a context");
    cudaStream_t st = (cudaStream_t)stream;
    if (B > 0) {
        const int64_t Bc = flow_chunk_rows(f, B, ws_bytes, 1);
        ZK_REQUIRE(Bc > 0, "flow_log_prob: workspace too small (%zu < %zu)", ws_bytes, zk_flow_min_workspace_bytes(f));
        for (int64_t i0 = 0; i0 < B; i0 += Bc) {
            const int64_t n = std::min(Bc, B - i0);
            ZK_TRY(flow_forward_chunk(f, x + i0 * ldx, ldx, c ? c + i0 * ldc : nullptr, ldc, n, nullptr, 0,
                                      nullptr, log_prob + i0, ws, ws_bytes, st));
        }
    }
    if (sum_log_prob) {
        ZK_REQUIRE(ws_bytes >= reduce_scratch_bytes(), "flow_log_prob: workspace too small for the reduction");
        ZK_TRY(launch_sum_f32_to_f64(log_prob, B, sum_log_prob, ws, st));
    }
    return ZK_OK;
}

zk_status zk_flow_inverse(const zk_flow_desc* f, const float* z, int64_t ldz, const float* c,
                          int64_t ldc, int64_t B, float* x, int64_t ldx, float* log_prob, void* ws,
                          size_t ws_bytes, zk_stream stream) {
    ZK_TRY(flow_check(f));
    ZK_REQUIRE(x && z, "flow_inverse: null argument");
    ZK_REQUIRE(x != z, "flow_inverse: x must not alias z");
    ZK_REQUIRE(B >= 0 && ldx >= f->features && ldz >= f->features, "flow_inverse: bad shape");
    ZK_REQUIRE(f->context == 0 || c, "flow_inverse: flow needs a context");
    if (B == 0) return ZK_OK;
    const int64_t Bc = flow_chunk_rows(f, B, ws_bytes, 2);
    ZK_REQUIRE(Bc > 0, "flow_inverse: workspace too small (%zu < %zu)", ws_bytes, zk_flow_min_workspace_bytes(f));
    for (int64_t i0 = 0; i0 < B; i0 += Bc) {
        const int64_t n = std::min(Bc, B - i0);
        ZK_TRY(flow_inverse_chunk(f, z + i0 * ldz, ldz, c ? c + i0 * ldc : nullptr, ldc, n, x + i0 * ldx,
                                  ldx, log_prob ? log_prob + i0 : nullptr, ws, ws_bytes,
                                  (cudaStream_t)stream));
    }
    return ZK_OK;
}

// ---------------------------------------------------------------------------
// host-buffer entry point: H2D | compute | D2H pipelined over row chunks
// ---------------------------------------------------------------------------
namespace zkapi {
struct HostPipe {
    cudaStream_t h2d = nullptr, d2h = nullptr;
    cudaEvent_t ev_h2d[2] = {nullptr, nullptr}, ev_comp[2] = {nullptr, nullptr}, ev_d2h[2] = {nullptr, nullptr};
    bool ready = false;
};
HostPipe g_pipe[64];
std::mutex g_pipe_mu;

zk_status get_pipe(HostPipe** out) {
    int dev = 0;
    ZK_CUDA(cudaGetDevice(&dev));
    ZK_REQUIRE(dev >= 0 && dev < 64, "device index out of range");
    std::lock_guard<std::mutex> lk(g_pipe_mu);
    HostPipe& p = g_pipe[dev];
    if (!p.ready) {
        ZK_CUDA(cudaStreamCreateWithFlags(&p.h2d, cudaStreamNonBlocking));
        ZK_CUDA(cudaStreamCreateWithFlags(&p.d2h, cudaStreamNonBlocking));
        for (int i = 0; i < 2; ++i) {
            ZK_CUDA(cudaEventCreateWithFlags(&p.ev_h2d[i], cudaEventDisableTiming));
            ZK_CUDA(cudaEventCreateWithFlags(&p.ev_comp[i], cudaEventDisableTiming));
            ZK_CUDA(cudaEventCreateWithFlags(&p.ev_d2h[i], cudaEventDisableTiming));
        }
        p.ready = true;
    }
    *out = &p;
    return ZK_OK;
}
}  // namespace zkapi

}  // extern "C"

/* Row chunks of the host pipeline.  The H2D copies run ahead of the compute (47 GB/s against ~30 GB/s of
   input consumed by cfg2, less for every heavier flow), so a call costs copy(first chunk) + compute(all) +
   a per-launch ramp per chunk: the first chunk is ONE wave of the persistent kernels (a wave = SMs/2 CTA pairs x
   512 rows; chunks are whole waves, a 3.46-wave chunk runs as 4), the later ones grow by <= 1.7x — with two
   staging slots the copy of chunk k starts when chunk k-2 is done and has to finish within the compute of
   chunk k-1 — up to `max_chunk` (what the workspace holds).  Small batches: eight equal chunks as before. */
std::vector<int64_t> host_chunk_plan(int64_t B, int64_t wave, int64_t max_chunk) {
    std::vector<int64_t> plan;
    if (B <= 0) return plan;
    max_chunk = std::max<int64_t>(1, max_chunk);
    if (B <= 4 * wave || max_chunk < wave) {
        const int64_t Bc = std::min(std::min(max_chunk, B), std::max<int64_t>(4096, ceil_div(B, 8)));
        for (int64_t i = 0; i < B; i += Bc) plan.push_back(std::min(Bc, B - i));
        return plan;
    }
    const int64_t cap = std::max<int64_t>(wave, (max_chunk / wave) * wave);
    int64_t left = B, w = 1;  // w: next chunk in waves
    while (left > 0) {
        int64_t n = std::min(std::min(w * wave, cap), left);
        if (left - n < wave / 2 && left <= cap) n = left;  // a sliver is not worth its own launches
        plan.push_back(n);
        left -= n;
        w = std::min<int64_t>(32, (w * 3 + 1) / 2);  // 1 2 3 5 8 12 18 27 32 32 ...: past ~1 M rows a chunk's ramp is noise, its staging is not
    }
    return plan;
}

static size_t host_pipe_need(const zk_flow_desc* f, int64_t n) {
    const size_t D = (size_t)f->features, C = (size_t)f->context;
    return 2 * (a256((size_t)n * D * 4) + a256((size_t)n * C * 4) + a256((size_t)n * 4)) + a256(C * 4) +
           a256(4096 * sizeof(double)) + flow_ws_for(f, n);
}

extern "C" {

size_t zk_flow_host_workspace_bytes(const zk_flow_desc* f, int64_t B) {
    if (!f || B <= 0) return 1024;
    const int64_t wave = (int64_t)(sm_count() / 2) * 512;
    int64_t big = 0;
    for (int64_t n : host_chunk_plan(B, wave, B)) big = std::max(big, n);
    return host_pipe_need(f, big) + 4096;
}

int64_t zk_debug_host_chunk_plan(int64_t B, int64_t wave, int64_t max_chunk, int64_t* out, int64_t cap) {
    const std::vector<int64_t> plan = host_chunk_plan(B, wave, max_chunk);
    for (size_t i = 0; i < plan.size() && (int64_t)i < cap; ++i) out[i] = plan[i];
    return (int64_t)plan.size();
}

zk_status zk_flow_log_prob_host(const zk_flow_desc* f, const float* xh, int64_t ldx, const float* ch,
                                int64_t ldc, int64_t B, float* lph, double* sum_host, void* ws,
                                size_t ws_bytes, zk_stream stream) {
    ZK_TRY(flow_check(f));
    ZK_REQUIRE(xh && lph, "flow_log_prob_host: null argument");
    ZK_REQUIRE(B >= 0 && ldx >= f->features, "flow_log_prob_host: bad shape");
    ZK_REQUIRE(f->context == 0 || ch, "flow_log_prob_host: flow needs a context");
    ZK_REQUIRE(ldc == 0 || ldc >= f->context, "flow_log_prob_host: bad ldc");
    if (sum_host) *sum_host = 0.0;
    if (B == 0) return ZK_OK;
    cudaStream_t st = (cudaStream_t)stream;
    HostPipe* pp = nullptr;
    ZK_TRY(get_pipe(&pp));
    HostPipe& p = *pp;
    const int D = f->features, C = f->context;
    const bool bc = (C > 0 && ldc == 0);  // one broadcast context row
    // staging per row: x + c + lp, two slots; the rest of the workspace runs the flow
    const size_t stage_row = (size_t)(D + (bc ? 0 : C) + 1) * 4;
    // chunk plan (host_chunk_plan): the step's time is the FIRST chunk's copy plus the compute of all of them,
    // so the first chunk is one wave and the later ones grow; bounded by the workspace
    const int64_t wave = (int64_t)(sm_count() / 2) * 512;
    auto need = [&](int64_t n) { return host_pipe_need(f, n); };
    int64_t Bmax = B;
    while (Bmax > 1 && need(Bmax) > ws_bytes) Bmax = (Bmax > wave) ? std::max<int64_t>(wave, (Bmax / 2 / wave) * wave) : (Bmax + 1) / 2;
    ZK_REQUIRE(need(Bmax) <= ws_bytes, "flow_log_prob_host: workspace too small (%zu < %zu)", ws_bytes, need(1));
    (void)stage_row;
    const std::vector<int64_t> plan = host_chunk_plan(B, wave, Bmax);
    const int64_t nchunks = (int64_t)plan.size();
    ZK_REQUIRE(nchunks <= 4096, "flow_log_prob_host: too many chunks; pass a larger workspace");
    int64_t Bc = 0;
    for (int64_t n : plan) Bc = std::max(Bc, n);
    Arena ar(ws, ws_bytes);
    float* xd[2] = {ar.take<float>((size_t)Bc * D), ar.take<float>((size_t)Bc * D)};
    float* cd[2] = {nullptr, nullptr};
    float* cb = nullptr;
    if (C > 0 && !bc) { cd[0] = ar.take<float>((size_t)Bc * C); cd[1] = ar.take<float>((size_t)Bc * C); }
    if (bc) cb = ar.take<float>((size_t)C);
    float* lpd[2] = {ar.take<float>((size_t)Bc), ar.take<float>((size_t)Bc)};
    double* sums = ar.take<double>(4096);
    ZK_REQUIRE(ar.ok, "flow_log_prob_host: workspace too small");
    void* fws = ar.base + ar.off;
    const size_t fws_bytes = ar.size - ar.off;

    // order the side streams after the caller's stream
    ZK_CUDA(cudaEventRecord(p.ev_comp[0], st));
    ZK_CUDA(cudaStreamWaitEvent(p.h2d, p.ev_comp[0], 0));
    ZK_CUDA(cudaStreamWaitEvent(p.d2h, p.ev_comp[0], 0));
    if (bc) ZK_CUDA(cudaMemcpyAsync(cb, ch, (size_t)C * 4, cudaMemcpyHostToDevice, p.h2d));
    int64_t i0 = 0;
    for (int64_t k = 0; k < nchunks; i0 += plan[(size_t)k], ++k) {
        const int s = (int)(k & 1);
        const int64_t n = plan[(size_t)k];
        if (k >= 2) {  // slot reuse: chunk k-2 must have been computed and read back
            ZK_CUDA(cudaStreamWaitEvent(p.h2d, p.ev_comp[s], 0));
        }
        if (ldx == D) {
            ZK_CUDA(cudaMemcpyAsync(xd[s], xh + i0 * ldx, (size_t)n * D * 4, cudaMemcpyHostToDevice, p.h2d));
        } else {
            ZK_CUDA(cudaMemcpy2DAsync(xd[s], (size_t)D * 4, xh + i0 * ldx, (size_t)ldx * 4, (size_t)D * 4, (size_t)n, cudaMemcpyHostToDevice, p.h2d));
        }
        if (C > 0 && !bc) {
            if (ldc == C) {
                ZK_CUDA(cudaMemcpyAsync(cd[s], ch + i0 * ldc, (size_t)n * C * 4, cudaMemcpyHostToDevice, p.h2d));
            } else {
                ZK_CUDA(cudaMemcpy2DAsync(cd[s], (size_t)C * 4, ch + i0 * ldc, (size_t)ldc * 4, (size_t)C * 4, (size_t)n, cudaMemcpyHostToDevice, p.h2d));
            }
        }
        ZK_CUDA(cudaEventRecord(p.ev_h2d[s], p.h2d));
        ZK_CUDA(cudaStreamWaitEvent(st, p.ev_h2d[s], 0));
        if (k >= 2) ZK_CUDA(cudaStreamWaitEvent(st, p.ev_d2h[s], 0));  // lpd[s] free again
        const float* cptr = C == 0 ? nullptr : (bc ? cb : cd[s]);
        ZK_TRY(flow_forward_chunk(f, xd[s], D, cptr, bc ? 0 : C, n, nullptr, 0, nullptr, lpd[s], fws, fws_bytes, st));
        if (sum_host) ZK_TRY(launch_sum_f32_to_f64(lpd[s], n, sums + k, fws, st));
        ZK_CUDA(cudaEventRecord(p.ev_comp[s], st));
        ZK_CUDA(cudaStreamWaitEvent(p.d2h, p.ev_comp[s], 0));
        ZK_CUDA(cudaMemcpyAsync(lph + i0, lpd[s], (size_t)n * 4, cudaMemcpyDeviceToHost, p.d2h));
        ZK_CUDA(cudaEventRecord(p.ev_d2h[s], p.d2h));
    }
    std::vector<double> hs;
    if (sum_host) {
        hs.resize((size_t)nchunks);
        ZK_CUDA(cudaMemcpyAsync(hs.data(), sums, (size_t)nchunks * sizeof(double), cudaMemcpyDeviceToHost, st));
    }
    ZK_CUDA(cudaStreamSynchronize(p.d2h));
    ZK_CUDA(cudaStreamSynchronize(st));
    if (sum_host) {
        double acc = 0.0;
        for (double v : hs) acc += v;  // fixed chunk order
        *sum_host = acc;
    }
    return ZK_OK;
}

}  // extern "C"
