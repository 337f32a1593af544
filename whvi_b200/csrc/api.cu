// extern "C" surface of libwhvi_b200.so (declared in include/whvi_b200.h): argument
// validation, error text, dispatch to the launchers.  Nothing here allocates or syncs.
#include "common.cuh"

namespace whvi {
char* error_buffer()
{
    static thread_local char buf[512] = {0};
    return buf;
}
}  // namespace whvi

using namespace whvi;

extern "C" {

int whvi_abi_version(void) { return WHVI_ABI_VERSION; }

const char* whvi_last_error(void) { return error_buffer(); }

int64_t whvi_max_dim(void) { return int64_t(1) << kMaxLog2Dmulti; }

int whvi_fwht_f32(const float* in, float* out, int64_t rows, int64_t D, whvi_stream_t stream)
{
    if (rows < 0 || D < 1) return fail(WHVI_E_SHAPE, "fwht: rows=%lld D=%lld", (long long)rows, (long long)D);
    if (!is_pow2(D)) return fail(WHVI_E_SHAPE, "fwht: n must be a power of 2 (got %lld)", (long long)D);
    if (rows == 0) return WHVI_OK;
    if (!in || !out) return fail(WHVI_E_NULL, "fwht: null pointer");
    if (!aligned16(in) || !aligned16(out)) return fail(WHVI_E_ALIGN, "fwht: pointers must be 16-byte aligned");
    return launch_fwht(in, out, rows, D, static_cast<cudaStream_t>(stream));
}

int whvi_fwht_scaled_f32(const float* in, const float* scale, float* out, int64_t rows, int64_t D, whvi_stream_t stream)
{
    if (rows < 0 || D < 4) return fail(WHVI_E_SHAPE, "fwht_scaled: rows=%lld D=%lld (D >= 4)", (long long)rows, (long long)D);
    if (!is_pow2(D)) return fail(WHVI_E_SHAPE, "fwht_scaled: n must be a power of 2 (got %lld)", (long long)D);
    if (rows == 0) return WHVI_OK;
    if (!in || !scale || !out) return fail(WHVI_E_NULL, "fwht_scaled: null pointer");
    if (!aligned16(in) || !aligned16(out) || !aligned16(scale)) return fail(WHVI_E_ALIGN, "fwht_scaled: pointers must be 16-byte aligned");
    return launch_fwht_scaled(in, scale, out, rows, D, static_cast<cudaStream_t>(stream));
}

int whvi_fwht_bf16(const void* in, void* out, int64_t rows, int64_t D, whvi_stream_t stream)
{
    if (rows < 0 || D < 1) return fail(WHVI_E_SHAPE, "fwht_bf16: rows=%lld D=%lld", (long long)rows, (long long)D);
    if (!is_pow2(D)) return fail(WHVI_E_SHAPE, "fwht_bf16: n must be a power of 2 (got %lld)", (long long)D);
    if (rows == 0) return WHVI_OK;
    if (!in || !out) return fail(WHVI_E_NULL, "fwht_bf16: null pointer");
    if ((reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(out)) & 7u) return fail(WHVI_E_ALIGN, "fwht_bf16: pointers must be 8-byte aligned");
    return launch_fwht_bf16(in, out, rows, D, static_cast<cudaStream_t>(stream));
}

int whvi_fwht_f64(const double* in, double* out, int64_t rows, int64_t D, whvi_stream_t stream)
{
    if (rows < 0 || D < 1) return fail(WHVI_E_SHAPE, "fwht_f64: rows=%lld D=%lld", (long long)rows, (long long)D);
    if (!is_pow2(D)) return fail(WHVI_E_SHAPE, "fwht_f64: n must be a power of 2 (got %lld)", (long long)D);
    if (rows == 0) return WHVI_OK;
    if (!in || !out) return fail(WHVI_E_NULL, "fwht_f64: null pointer");
    if (!aligned16(in) || !aligned16(out)) return fail(WHVI_E_ALIGN, "fwht_f64: pointers must be 16-byte aligned");
    if (rows > (int64_t(1) << 40) / D) return fail(WHVI_E_SHAPE, "fwht_f64: too many elements");
    return launch_fwht_f64(in, out, rows, D, static_cast<cudaStream_t>(stream));
}

static int check_layer_shape(const char* who, int64_t S, int64_t B, int64_t D, int64_t xs, int64_t max_d = 8192)
{
    if (S < 0 || B < 0 || D < 1) return fail(WHVI_E_SHAPE, "%s: S=%lld B=%lld D=%lld", who, (long long)S, (long long)B, (long long)D);
    if (!is_pow2(D)) return fail(WHVI_E_SHAPE, "%s: D must be a power of 2 (got %lld)", who, (long long)D);
    if (D < 4 || D > max_d) return fail(WHVI_E_SHAPE, "%s: D = %lld outside [4, %lld]", who, (long long)D, (long long)max_d);
    if (xs != 0 && xs != B * D) return fail(WHVI_E_SHAPE, "%s: x_sample_stride must be 0 or B*D", who);
    return WHVI_OK;
}

int whvi_layer_fwd_partials(int64_t S, int64_t B, int64_t D, int64_t* count)
{
    if (!count) return fail(WHVI_E_NULL, "layer_fwd_partials: null pointer");
    if (int rc = check_layer_shape("layer_fwd_partials", S, B, D, 0, 32768)) return rc;
    *count = 0;
    if (S == 0 || B == 0) return WHVI_OK;
    size_t n = 0;
    LayerFwdCall c{};
    c.S = S;
    c.B = B;
    c.partials_needed = &n;
    const int rc = launch_layer_fwd(c, D, nullptr);
    *count = static_cast<int64_t>(n);
    return rc;
}

int whvi_layer_fwd_fused_f32(const float* x, int64_t x_sample_stride, const float* g, const float* s1, const float* s2,
                             const float* bias, float* y, int64_t S, int64_t B, int64_t D, int flags,
                             const float* target, float* sq_partials, whvi_stream_t stream)
{
    if (int rc = check_layer_shape("layer_fwd", S, B, D, x_sample_stride, 32768)) return rc;
    if (flags & ~(WHVI_LAYER_RELU_OUT | WHVI_LAYER_FROM_T2)) return fail(WHVI_E_MODE, "layer_fwd: unknown flags %d", flags);
    if (S == 0 || B == 0) return WHVI_OK;
    if (!x || !g || !s1 || !s2 || !y) return fail(WHVI_E_NULL, "layer_fwd: null pointer");
    if (target && !sq_partials) return fail(WHVI_E_NULL, "layer_fwd: target given without sq_partials");
    if (!aligned16(x) || !aligned16(g) || !aligned16(s1) || !aligned16(s2) || !aligned16(y) || !aligned16(bias) ||
        !aligned16(target))
        return fail(WHVI_E_ALIGN, "layer_fwd: pointers must be 16-byte aligned");
    LayerFwdCall c{x, g, s1, s2, bias, target, y, sq_partials, x_sample_stride, S, B, flags & WHVI_LAYER_RELU_OUT, nullptr};
    c.from_t2 = (flags & WHVI_LAYER_FROM_T2) ? 1 : 0;
    return launch_layer_fwd(c, D, static_cast<cudaStream_t>(stream));
}

int whvi_layer_fwd_bf16(const void* x, int64_t x_sample_stride, const float* g, const float* s1, const float* s2, const float* bias,
                        void* y, int64_t S, int64_t B, int64_t D, int flags, whvi_stream_t stream)
{
    if (int rc = check_layer_shape("layer_fwd_bf16", S, B, D, x_sample_stride, 32768)) return rc;
    if (flags & ~(WHVI_LAYER_RELU_OUT | WHVI_LAYER_FROM_T2)) return fail(WHVI_E_MODE, "layer_fwd_bf16: unknown flags %d", flags);
    if (S == 0 || B == 0) return WHVI_OK;
    if (!x || !g || !s1 || !s2 || !y) return fail(WHVI_E_NULL, "layer_fwd_bf16: null pointer");
    if (!aligned16(g) || !aligned16(s1) || !aligned16(s2) || !aligned16(bias) ||
        ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 7u))
        return fail(WHVI_E_ALIGN, "layer_fwd_bf16: fp32 pointers must be 16-byte aligned, bf16 pointers 8-byte aligned");
    LayerFwdCall c{static_cast<const float*>(x), g, s1, s2, bias, nullptr, static_cast<float*>(y), nullptr, x_sample_stride, S, B,
                   flags & WHVI_LAYER_RELU_OUT, nullptr};
    c.from_t2 = (flags & WHVI_LAYER_FROM_T2) ? 1 : 0;
    c.bf16 = 1;
    return launch_layer_fwd(c, D, static_cast<cudaStream_t>(stream));
}

int whvi_layer_fwd_f32(const float* x, int64_t x_sample_stride, const float* g, const float* s1, const float* s2,
                       const float* bias, float* y, int64_t S, int64_t B, int64_t D, whvi_stream_t stream)
{
    return whvi_layer_fwd_fused_f32(x, x_sample_stride, g, s1, s2, bias, y, S, B, D, 0, nullptr, nullptr, stream);
}

int whvi_layer_bwd_workspace_bytes(int64_t S, int64_t B, int64_t D, size_t* bytes)
{
    if (!bytes) return fail(WHVI_E_NULL, "layer_bwd_workspace_bytes: null pointer");
    if (int rc = check_layer_shape("layer_bwd_workspace_bytes", S, B, D, 0)) return rc;
    *bytes = 0;
    if (S == 0 || B == 0) return WHVI_OK;
    LayerBwdCall c{};
    c.S = S;
    c.B = B;
    c.need_only = bytes;
    return launch_layer_bwd(c, D, nullptr);
}

static int layer_bwd_common(const float* x, int64_t x_sample_stride, const float* dy, const float* g, const float* s1,
                            const float* s2, float* dx, float* dg, float* ds1, float* ds2, float* dbias,
                            void* workspace, size_t workspace_bytes, int64_t S, int64_t B, int64_t D, int flags,
                            const float* target, const float* coef, const float* dy_scale, whvi_stream_t stream)
{
    if (int rc = check_layer_shape("layer_bwd", S, B, D, x_sample_stride)) return rc;
    if (flags & ~WHVI_LAYER_RELU_IN) return fail(WHVI_E_MODE, "layer_bwd: unknown flags %d", flags);
    if (!dg || !ds1 || !ds2) return fail(WHVI_E_NULL, "layer_bwd: null output pointer");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (S == 0 || B == 0) {  // empty sums
        if (S > 0) cudaMemsetAsync(dg, 0, sizeof(float) * size_t(S) * D, st);
        cudaMemsetAsync(ds1, 0, sizeof(float) * D, st);
        cudaMemsetAsync(ds2, 0, sizeof(float) * D, st);
        if (dbias) cudaMemsetAsync(dbias, 0, sizeof(float) * D, st);
        return check_launch("layer_bwd(empty)");
    }
    if (!x || !dy || !g || !s1 || !s2) return fail(WHVI_E_NULL, "layer_bwd: null pointer");
    if (target && !coef) return fail(WHVI_E_NULL, "layer_bwd: target given without coef");
    if (!aligned16(x) || !aligned16(dy) || !aligned16(g) || !aligned16(s1) || !aligned16(s2) || !aligned16(dx) ||
        !aligned16(workspace) || !aligned16(target))
        return fail(WHVI_E_ALIGN, "layer_bwd: pointers must be 16-byte aligned");
    LayerBwdCall c{x, dy, g, s1, s2, target, coef, nullptr, dx, dg, ds1, ds2, dbias, static_cast<float*>(workspace),
                   workspace_bytes, x_sample_stride, S, B, flags & WHVI_LAYER_RELU_IN, nullptr};
    c.dy_scale = dy_scale;
    return launch_layer_bwd(c, D, st);
}

int whvi_layer_bwd_fused_f32(const float* x, int64_t x_sample_stride, const float* dy, const float* g, const float* s1,
                             const float* s2, float* dx, float* dg, float* ds1, float* ds2, float* dbias,
                             void* workspace, size_t workspace_bytes, int64_t S, int64_t B, int64_t D, int flags,
                             const float* target, const float* coef, whvi_stream_t stream)
{
    return layer_bwd_common(x, x_sample_stride, dy, g, s1, s2, dx, dg, ds1, ds2, dbias, workspace, workspace_bytes, S, B, D,
                            flags, target, coef, nullptr, stream);
}

int whvi_layer_bwd_scaled_f32(const float* x, int64_t x_sample_stride, const float* dy, const float* dy_scale,
                              const float* g, const float* s1, const float* s2, float* dx, float* dg, float* ds1,
                              float* ds2, float* dbias, void* workspace, size_t workspace_bytes, int64_t S, int64_t B,
                              int64_t D, int flags, whvi_stream_t stream)
{
    return layer_bwd_common(x, x_sample_stride, dy, g, s1, s2, dx, dg, ds1, ds2, dbias, workspace, workspace_bytes, S, B, D,
                            flags, nullptr, nullptr, dy_scale, stream);
}

// bf16 activations (x, dy, dx): the fp32 kernels' plan on widened tiles, dx rounded once at the store.  x and dy arrive by
// bulk async copies, which need 16-byte-aligned addresses and sizes: with 2-byte elements a sample (B * D elements) and the
// tail tile of a sample are whole 16-byte units only when B * D % 8 == 0 (it fails only at D = 4 with an odd B).
static int check_bf16_io(const char* who, const void* x, const void* dy, const void* dx, int64_t B, int64_t D)
{
    if ((B * D) % 8 != 0)
        return fail(WHVI_E_SHAPE, "%s: B * D = %lld must be a multiple of 8 for bf16 activations (pad B)", who, (long long)(B * D));
    if (!aligned16(x) || !aligned16(dy) || (reinterpret_cast<uintptr_t>(dx) & 7u))
        return fail(WHVI_E_ALIGN, "%s: x and dy must be 16-byte aligned, dx 8-byte aligned", who);
    return WHVI_OK;
}

int whvi_layer_bwd_bf16(const void* x, int64_t x_sample_stride, const void* dy, const float* dy_scale, const float* g,
                        const float* s1, const float* s2, void* dx, float* dg, float* ds1, float* ds2, float* dbias,
                        void* workspace, size_t workspace_bytes, int64_t S, int64_t B, int64_t D, int flags, whvi_stream_t stream)
{
    if (int rc = check_layer_shape("layer_bwd_bf16", S, B, D, x_sample_stride)) return rc;
    if (flags & ~WHVI_LAYER_RELU_IN) return fail(WHVI_E_MODE, "layer_bwd_bf16: unknown flags %d", flags);
    if (!dg || !ds1 || !ds2) return fail(WHVI_E_NULL, "layer_bwd_bf16: null output pointer");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (S == 0 || B == 0) {  // empty sums
        if (S > 0) cudaMemsetAsync(dg, 0, sizeof(float) * size_t(S) * D, st);
        cudaMemsetAsync(ds1, 0, sizeof(float) * D, st);
        cudaMemsetAsync(ds2, 0, sizeof(float) * D, st);
        if (dbias) cudaMemsetAsync(dbias, 0, sizeof(float) * D, st);
        return check_launch("layer_bwd_bf16(empty)");
    }
    if (!x || !dy || !g || !s1 || !s2) return fail(WHVI_E_NULL, "layer_bwd_bf16: null pointer");
    if (!aligned16(g) || !aligned16(s1) || !aligned16(s2) || !aligned16(workspace))
        return fail(WHVI_E_ALIGN, "layer_bwd_bf16: fp32 pointers must be 16-byte aligned");
    if (int rc = check_bf16_io("layer_bwd_bf16", x, dy, dx, B, D)) return rc;
    LayerBwdCall c{static_cast<const float*>(x), static_cast<const float*>(dy), g, s1, s2, nullptr, nullptr, dy_scale,
                   static_cast<float*>(dx), dg, ds1, ds2, dbias, static_cast<float*>(workspace), workspace_bytes, x_sample_stride, S, B,
                   flags & WHVI_LAYER_RELU_IN, nullptr};
    c.bf16 = 1;
    return launch_layer_bwd(c, D, st);
}

int whvi_layer_loss_sizes(int64_t S, int64_t B, int64_t D, size_t* workspace_bytes, int64_t* sq_count)
{
    if (!workspace_bytes || !sq_count) return fail(WHVI_E_NULL, "layer_loss_sizes: null pointer");
    if (int rc = check_layer_shape("layer_loss_sizes", S, B, D, 0, 4096)) return rc;
    if (D < 128) return fail(WHVI_E_SHAPE, "layer_loss: D = %lld outside [128, 4096]", (long long)D);
    *workspace_bytes = 0;
    *sq_count = 0;
    if (S == 0 || B == 0) return WHVI_OK;
    LayerLossCall c{};
    c.S = S;
    c.B = B;
    c.need_ws = workspace_bytes;
    c.need_sq = sq_count;
    return launch_layer_loss(c, D, nullptr);
}

int whvi_layer_loss_f32(const float* x, int64_t x_sample_stride, const float* g, const float* s1, const float* s2,
                        const float* bias, const float* target, float* dx, float* dg, float* ds1, float* ds2,
                        float* dbias, float* sq_partials, void* workspace, size_t workspace_bytes, int64_t S, int64_t B,
                        int64_t D, int flags, whvi_stream_t stream)
{
    if (int rc = check_layer_shape("layer_loss", S, B, D, x_sample_stride, 4096)) return rc;
    if (D < 128) return fail(WHVI_E_SHAPE, "layer_loss: D = %lld outside [128, 4096]", (long long)D);
    if (flags & ~WHVI_LAYER_RELU_IN) return fail(WHVI_E_MODE, "layer_loss: unknown flags %d", flags);
    if (S == 0 || B == 0) return fail(WHVI_E_SHAPE, "layer_loss: empty batch");
    if (!x || !g || !s1 || !s2 || !target || !dg || !ds1 || !ds2 || !sq_partials || (bias && !dbias))
        return fail(WHVI_E_NULL, "layer_loss: null pointer");
    if (!aligned16(x) || !aligned16(g) || !aligned16(s1) || !aligned16(s2) || !aligned16(bias) || !aligned16(target) ||
        !aligned16(dx) || !aligned16(workspace))
        return fail(WHVI_E_ALIGN, "layer_loss: pointers must be 16-byte aligned");
    LayerLossCall c{x, g, s1, s2, bias, target, dx, dg, ds1, ds2, dbias, sq_partials, static_cast<float*>(workspace),
                    workspace_bytes, x_sample_stride, S, B, flags & WHVI_LAYER_RELU_IN, nullptr, nullptr};
    return launch_layer_loss(c, D, static_cast<cudaStream_t>(stream));
}

int whvi_layer_loss_bf16(const void* x, int64_t x_sample_stride, const float* g, const float* s1, const float* s2,
                         const float* bias, const float* target, void* dx, float* dg, float* ds1, float* ds2, float* dbias,
                         float* sq_partials, void* workspace, size_t workspace_bytes, int64_t S, int64_t B, int64_t D, int flags,
                         whvi_stream_t stream)
{
    if (int rc = check_layer_shape("layer_loss_bf16", S, B, D, x_sample_stride, 4096)) return rc;
    if (D < 128) return fail(WHVI_E_SHAPE, "layer_loss_bf16: D = %lld outside [128, 4096]", (long long)D);
    if (flags & ~WHVI_LAYER_RELU_IN) return fail(WHVI_E_MODE, "layer_loss_bf16: unknown flags %d", flags);
    if (S == 0 || B == 0) return fail(WHVI_E_SHAPE, "layer_loss_bf16: empty batch");
    if (!x || !g || !s1 || !s2 || !target || !dg || !ds1 || !ds2 || !sq_partials || (bias && !dbias))
        return fail(WHVI_E_NULL, "layer_loss_bf16: null pointer");
    if (!aligned16(g) || !aligned16(s1) || !aligned16(s2) || !aligned16(bias) || !aligned16(target) || !aligned16(workspace))
        return fail(WHVI_E_ALIGN, "layer_loss_bf16: fp32 pointers must be 16-byte aligned");
    if (!aligned16(x) || (reinterpret_cast<uintptr_t>(dx) & 7u))
        return fail(WHVI_E_ALIGN, "layer_loss_bf16: x must be 16-byte aligned, dx 8-byte aligned");
    LayerLossCall c{static_cast<const float*>(x), g, s1, s2, bias, target, static_cast<float*>(dx), dg, ds1, ds2, dbias, sq_partials,
                    static_cast<float*>(workspace), workspace_bytes, x_sample_stride, S, B, flags & WHVI_LAYER_RELU_IN, nullptr, nullptr};
    c.bf16 = 1;
    return launch_layer_loss(c, D, static_cast<cudaStream_t>(stream));
}

int whvi_layer_bwd_f32(const float* x, int64_t x_sample_stride, const float* dy, const float* g, const float* s1,
                       const float* s2, float* dx, float* dg, float* ds1, float* ds2, float* dbias, void* workspace,
                       size_t workspace_bytes, int64_t S, int64_t B, int64_t D, whvi_stream_t stream)
{
    return whvi_layer_bwd_fused_f32(x, x_sample_stride, dy, g, s1, s2, dx, dg, ds1, ds2, dbias, workspace,
                                    workspace_bytes, S, B, D, 0, nullptr, nullptr, stream);
}

int whvi_reparam_f32(const float* mu, const float* rho, const float* eps, float* g, int64_t S, int64_t D, int mode,
                     whvi_stream_t stream)
{
    if (S < 0 || D < 1) return fail(WHVI_E_SHAPE, "reparam: S=%lld D=%lld", (long long)S, (long long)D);
    if (mode != WHVI_REPARAM_DIAG && mode != WHVI_REPARAM_DENSE) return fail(WHVI_E_MODE, "reparam: unknown mode %d", mode);
    if (S == 0) return WHVI_OK;
    if (!mu || !rho || !eps || !g) return fail(WHVI_E_NULL, "reparam: null pointer");
    if (mode == WHVI_REPARAM_DENSE)
        return fail(WHVI_E_MODE, "reparam: the dense form needs a workspace -- call whvi_reparam_dense_f32");
    return launch_reparam_diag(mu, rho, eps, g, S, D, static_cast<cudaStream_t>(stream));
}

int whvi_reparam_dense_workspace_bytes(int64_t S, int64_t D, size_t* bytes)
{
    if (!bytes) return fail(WHVI_E_NULL, "reparam_dense_workspace_bytes: null pointer");
    if (S < 0 || D < 128 || D % 128 != 0) return fail(WHVI_E_SHAPE, "reparam(dense): S=%lld, D=%lld (D must be a multiple of 128)", (long long)S, (long long)D);
    *bytes = reparam_dense_workspace_bytes(S, D);
    return WHVI_OK;
}

int whvi_reparam_dense_f32(const float* mu, const float* L, const float* eps, float* g, int64_t S, int64_t D, void* workspace,
                           size_t workspace_bytes, whvi_stream_t stream)
{
    if (S < 0 || D < 128 || D % 128 != 0) return fail(WHVI_E_SHAPE, "reparam(dense): S=%lld, D=%lld (D must be a multiple of 128)", (long long)S, (long long)D);
    if (S == 0) return WHVI_OK;
    if (!mu || !L || !eps || !g) return fail(WHVI_E_NULL, "reparam(dense): null pointer");
    if (!aligned16(L) || !aligned16(eps) || !aligned16(workspace)) return fail(WHVI_E_ALIGN, "reparam(dense): pointers must be 16-byte aligned");
    return launch_reparam_dense(mu, L, eps, g, S, D, static_cast<float*>(workspace), workspace_bytes, static_cast<cudaStream_t>(stream));
}

int whvi_reparam_dense_bwd_f32(const float* dgT, const float* epsT, float* dL, int64_t S_padded, int64_t D, whvi_stream_t stream)
{
    if (S_padded <= 0 || S_padded % 32 != 0 || D < 128 || D % 128 != 0)
        return fail(WHVI_E_SHAPE, "reparam_bwd(dense): S_padded=%lld (multiple of 32), D=%lld (multiple of 128)", (long long)S_padded, (long long)D);
    if (!dgT || !epsT || !dL) return fail(WHVI_E_NULL, "reparam_bwd(dense): null pointer");
    if (!aligned16(dgT) || !aligned16(epsT) || !aligned16(dL)) return fail(WHVI_E_ALIGN, "reparam_bwd(dense): pointers must be 16-byte aligned");
    return launch_reparam_dense_bwd(dgT, epsT, dL, S_padded, D, static_cast<cudaStream_t>(stream));
}

int whvi_kl_dense_f32(const float* mu, const float* L, float lambda_, int64_t D, float* out_kl, float* dmu, float* dL, float grad_scale,
                      void* workspace, size_t workspace_bytes, whvi_stream_t stream)
{
    if (D < 1) return fail(WHVI_E_SHAPE, "kl(dense): D=%lld", (long long)D);
    if (!(lambda_ > 0.f)) return fail(WHVI_E_SHAPE, "kl(dense): lambda must be positive");
    if (!mu || !L || !out_kl) return fail(WHVI_E_NULL, "kl(dense): null pointer");
    if ((dmu == nullptr) != (dL == nullptr)) return fail(WHVI_E_NULL, "kl(dense): dmu and dL must both be given or both NULL");
    if (!workspace || workspace_bytes < sizeof(double) * size_t(D) || (reinterpret_cast<uintptr_t>(workspace) & 7u))
        return fail(WHVI_E_WORKSPACE, "kl(dense): workspace of %zu bytes (8-byte aligned) needed", sizeof(double) * size_t(D));
    return launch_kl_dense(mu, L, lambda_, D, out_kl, dmu, dL, grad_scale, static_cast<double*>(workspace), static_cast<cudaStream_t>(stream));
}

static int check_dense_grouped(const char* who, int64_t S, int64_t D, int64_t G, int64_t mu_stride, int64_t L_stride)
{
    if (S < 0 || D < 1 || G < 1 || (D > 64 && D % 128 != 0))
        return fail(WHVI_E_SHAPE, "%s: S=%lld D=%lld G=%lld (D <= 64 or a multiple of 128)", who, (long long)S, (long long)D, (long long)G);
    if (G > 65535) return fail(WHVI_E_SHAPE, "%s: G=%lld above 65535", who, (long long)G);
    if (G > 1 && (mu_stride < D || L_stride < D * D))
        return fail(WHVI_E_SHAPE, "%s: mu_stride=%lld must be >= D and L_stride=%lld >= D * D", who, (long long)mu_stride, (long long)L_stride);
    if (D >= 128 && G > 1 && (mu_stride % 4 != 0 || L_stride % 4 != 0))
        return fail(WHVI_E_SHAPE, "%s: strides must be multiples of 4 at D >= 128", who);
    if (S * G > 0x7fffffffLL) return fail(WHVI_E_SHAPE, "%s: too many samples", who);
    return WHVI_OK;
}

int whvi_reparam_dense_grouped_workspace_bytes(int64_t S, int64_t D, size_t* bytes)
{
    if (!bytes) return fail(WHVI_E_NULL, "reparam_dense_grouped_workspace_bytes: null pointer");
    if (int rc = check_dense_grouped("reparam_dense_grouped_workspace_bytes", S, D, 1, D, D * D)) return rc;
    *bytes = reparam_dense_grouped_workspace_bytes(S, D);
    return WHVI_OK;
}

int whvi_reparam_dense_grouped_f32(const float* mu, int64_t mu_stride, const float* L, int64_t L_stride, const float* eps, float* g, int64_t S,
                                   int64_t D, int64_t G, void* workspace, size_t workspace_bytes, whvi_stream_t stream)
{
    if (int rc = check_dense_grouped("reparam_dense_grouped", S, D, G, mu_stride, L_stride)) return rc;
    if (S == 0) return WHVI_OK;
    if (!mu || !L || !eps || !g) return fail(WHVI_E_NULL, "reparam_dense_grouped: null pointer");
    if (D >= 128) {
        if (!aligned16(L) || !aligned16(eps) || !aligned16(workspace))
            return fail(WHVI_E_ALIGN, "reparam_dense_grouped: L, eps and the workspace must be 16-byte aligned at D >= 128");
        if (!workspace || workspace_bytes < reparam_dense_grouped_workspace_bytes(S, D))
            return fail(WHVI_E_WORKSPACE, "reparam_dense_grouped: workspace of %zu bytes needed, %zu given", reparam_dense_grouped_workspace_bytes(S, D),
                        workspace_bytes);
    }
    return launch_reparam_dense_grouped(mu, mu_stride, L, L_stride, eps, g, S, D, G, static_cast<float*>(workspace), workspace_bytes,
                                        static_cast<cudaStream_t>(stream));
}

int whvi_reparam_dense_grouped_bwd_f32(const float* eps, const float* dg, float* dmu, float* dL, int64_t S, int64_t D, int64_t G, void* workspace,
                                       size_t workspace_bytes, whvi_stream_t stream)
{
    if (int rc = check_dense_grouped("reparam_dense_grouped_bwd", S, D, G, D, D * D)) return rc;
    if (!dmu || !dL) return fail(WHVI_E_NULL, "reparam_dense_grouped_bwd: null output pointer");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (S == 0) {
        cudaMemsetAsync(dmu, 0, sizeof(float) * size_t(G) * D, st);
        cudaMemsetAsync(dL, 0, sizeof(float) * size_t(G) * D * D, st);
        return check_launch("reparam_dense_grouped_bwd(empty)");
    }
    if (!eps || !dg) return fail(WHVI_E_NULL, "reparam_dense_grouped_bwd: null pointer");
    if (D >= 128) {
        if (!aligned16(dL) || !aligned16(workspace))
            return fail(WHVI_E_ALIGN, "reparam_dense_grouped_bwd: dL and the workspace must be 16-byte aligned at D >= 128");
        if (!workspace || workspace_bytes < reparam_dense_grouped_workspace_bytes(S, D))
            return fail(WHVI_E_WORKSPACE, "reparam_dense_grouped_bwd: workspace of %zu bytes needed, %zu given",
                        reparam_dense_grouped_workspace_bytes(S, D), workspace_bytes);
    }
    return launch_reparam_dense_grouped_bwd(eps, dg, dmu, dL, S, D, G, static_cast<float*>(workspace), workspace_bytes, st);
}

int whvi_kl_dense_grouped_f32(const float* mu, int64_t mu_stride, const float* L, int64_t L_stride, float lambda_, int64_t D, int64_t G,
                              float* out_kl, float* dmu, float* dL, float grad_scale, void* workspace, size_t workspace_bytes,
                              whvi_stream_t stream)
{
    if (D < 1 || D > 65535 || G < 1 || G > 65535 || (G > 1 && (mu_stride < D || L_stride < D * D)))
        return fail(WHVI_E_SHAPE, "kl_dense_grouped: D=%lld G=%lld mu_stride=%lld L_stride=%lld", (long long)D, (long long)G, (long long)mu_stride,
                    (long long)L_stride);
    if (!(lambda_ > 0.f)) return fail(WHVI_E_SHAPE, "kl_dense_grouped: lambda must be positive");
    if (!mu || !L || !out_kl) return fail(WHVI_E_NULL, "kl_dense_grouped: null pointer");
    if ((dmu == nullptr) != (dL == nullptr)) return fail(WHVI_E_NULL, "kl_dense_grouped: dmu and dL must both be given or both NULL");
    const size_t need = sizeof(double) * size_t(G) * size_t(D);
    if (!workspace || workspace_bytes < need || (reinterpret_cast<uintptr_t>(workspace) & 7u))
        return fail(WHVI_E_WORKSPACE, "kl_dense_grouped: workspace of %zu bytes (8-byte aligned) needed", need);
    return launch_kl_dense_grouped(mu, mu_stride, L, L_stride, lambda_, D, G, out_kl, dmu, dL, grad_scale, static_cast<double*>(workspace),
                                   static_cast<cudaStream_t>(stream));
}

int whvi_reparam_bwd_f32(const float* rho, const float* eps, const float* dg, float* dmu, float* drho, int64_t S,
                         int64_t D, int mode, int accumulate, whvi_stream_t stream)
{
    if (S < 0 || D < 1) return fail(WHVI_E_SHAPE, "reparam_bwd: S=%lld D=%lld", (long long)S, (long long)D);
    if (mode != WHVI_REPARAM_DIAG) return fail(WHVI_E_MODE, "reparam_bwd: unknown mode %d", mode);
    if (!rho || !dmu || !drho || (S > 0 && (!eps || !dg))) return fail(WHVI_E_NULL, "reparam_bwd: null pointer");
    return launch_reparam_diag_bwd(rho, eps, dg, dmu, drho, S, D, accumulate, static_cast<cudaStream_t>(stream));
}

int whvi_kl_f32(const float* mu, const float* rho, float lambda_, int64_t D, int mode, float* out_kl, float* dmu,
                float* drho, float grad_scale, int accumulate, whvi_stream_t stream)
{
    if (D < 1) return fail(WHVI_E_SHAPE, "kl: D=%lld", (long long)D);
    if (mode != WHVI_KL_REFERENCE && mode != WHVI_KL_CONSISTENT) return fail(WHVI_E_MODE, "kl: unknown mode %d", mode);
    if (!(lambda_ > 0.f)) return fail(WHVI_E_SHAPE, "kl: lambda must be positive");
    if (!mu || !rho || !out_kl) return fail(WHVI_E_NULL, "kl: null pointer");
    if ((dmu == nullptr) != (drho == nullptr)) return fail(WHVI_E_NULL, "kl: dmu and drho must both be given or both NULL");
    return launch_kl(mu, rho, lambda_, D, mode, out_kl, dmu, drho, grad_scale, accumulate, static_cast<cudaStream_t>(stream));
}

// ---- WHVIStackedMatrix as one call per direction (csrc/stacked.cu) ------------------------------------------------------
static int check_stacked(const char* who, int64_t S, int64_t B, int64_t D, int64_t G, int64_t n_out, int64_t xs, int64_t pstride)
{
    if (int rc = check_layer_shape(who, S, B, D, xs)) return rc;
    if (G < 1 || n_out <= (G - 1) * D || n_out > G * D)
        return fail(WHVI_E_SHAPE, "%s: G=%lld blocks of D=%lld do not match n_out=%lld", who, (long long)G, (long long)D, (long long)n_out);
    if (G > 65535) return fail(WHVI_E_SHAPE, "%s: G=%lld above 65535", who, (long long)G);   // the grouped reparam backward's grid.y
    if (G > 1 && (pstride < D || pstride % 4 != 0))
        return fail(WHVI_E_SHAPE, "%s: param_stride=%lld must be >= D and a multiple of 4", who, (long long)pstride);
    if (S * G > 0x7fffffffLL) return fail(WHVI_E_SHAPE, "%s: too many virtual samples", who);
    return WHVI_OK;
}

static int pad_rows(const char* who, const void* in, void* out, int64_t rows, int64_t n_in, int64_t D, int bf16, whvi_stream_t stream)
{
    if (rows < 0 || n_in < 1 || D < n_in || D % 4 != 0) return fail(WHVI_E_SHAPE, "%s: rows=%lld n_in=%lld D=%lld", who, (long long)rows, (long long)n_in, (long long)D);
    if (rows == 0) return WHVI_OK;
    if (!in || !out) return fail(WHVI_E_NULL, "%s: null pointer", who);
    if (!aligned16(out)) return fail(WHVI_E_ALIGN, "%s: out must be 16-byte aligned", who);
    if (bf16 && (reinterpret_cast<uintptr_t>(in) & 1u)) return fail(WHVI_E_ALIGN, "%s: in must be 2-byte aligned", who);
    return launch_stack_split(static_cast<const float*>(in), static_cast<float*>(out), rows, D, 1, n_in, static_cast<cudaStream_t>(stream), bf16);
}

int whvi_pad_rows_f32(const float* in, float* out, int64_t rows, int64_t n_in, int64_t D, whvi_stream_t stream)
{
    return pad_rows("pad_rows", in, out, rows, n_in, D, 0, stream);
}

int whvi_pad_rows_bf16(const void* in, void* out, int64_t rows, int64_t n_in, int64_t D, whvi_stream_t stream)
{
    return pad_rows("pad_rows_bf16", in, out, rows, n_in, D, 1, stream);
}

// bf16 activations (x, y_blocks, y, dy, dx) behind the float pointers of the internal calls: a pointer of 2-byte elements must be
// 2-byte aligned; the padded x and the block-layout dy of the backward arrive by bulk copy (see check_bf16_io)
static bool odd(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 1u) != 0; }

// the layer from g (G, S, D), however g was drawn; validated by the callers
static int stacked_fwd_g(const float* x, int64_t xs, const float* g, const float* s1, const float* s2, int64_t param_stride, const float* bias,
                         float* y_blocks, float* y, int64_t S, int64_t B, int64_t D, int64_t G, int64_t n_out, int flags, cudaStream_t st, int bf16 = 0)
{
    LayerFwdCall c{x, g, s1, s2, bias, nullptr, y_blocks, nullptr, xs, G * S, B, flags & WHVI_LAYER_RELU_OUT, nullptr};
    c.groups = G;
    c.pstride = param_stride;
    c.bstride = D;
    c.bf16 = bf16;
    if (int rc = launch_layer_fwd(c, D, st)) return rc;
    return launch_stack_concat(y_blocks, y, S * B, D, G, n_out, st, bf16);
}

// a Stacked forward: from (mu, rho, eps) drawn here, or -- from_g -- from g given (then mu, rho, eps are unused)
static int stacked_fwd(const char* who, int from_g, const void* x, int64_t x_sample_stride, const float* mu, const float* rho, const float* s1,
                       const float* s2, int64_t param_stride, const float* eps, const float* bias, float* g, void* y_blocks, void* y, int64_t S,
                       int64_t B, int64_t D, int64_t G, int64_t n_out, int flags, int bf16, whvi_stream_t stream)
{
    if (int rc = check_stacked(who, S, B, D, G, n_out, x_sample_stride, param_stride)) return rc;
    if (flags & ~WHVI_LAYER_RELU_OUT) return fail(WHVI_E_MODE, "%s: unknown flags %d", who, flags);
    if (S == 0 || B == 0) return WHVI_OK;
    if (!x || (!from_g && (!mu || !rho || !eps)) || !s1 || !s2 || !g || !y_blocks || !y) return fail(WHVI_E_NULL, "%s: null pointer", who);
    if (!aligned16(s1) || !aligned16(s2) || !aligned16(bias) || !aligned16(g))
        return fail(WHVI_E_ALIGN, "%s: pointers must be 16-byte aligned", who);
    if (bf16 ? ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y_blocks)) & 7u) || odd(y) : !aligned16(x) || !aligned16(y_blocks))
        return fail(WHVI_E_ALIGN, bf16 ? "%s: x and y_blocks must be 8-byte aligned, y 2-byte aligned" : "%s: pointers must be 16-byte aligned", who);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (!from_g)
        if (int rc = launch_reparam_diag(mu, rho, eps, g, G * S, D, st, G, param_stride)) return rc;
    return stacked_fwd_g(static_cast<const float*>(x), x_sample_stride, g, s1, s2, param_stride, bias, static_cast<float*>(y_blocks),
                         static_cast<float*>(y), S, B, D, G, n_out, flags, st, bf16);
}

int whvi_stacked_fwd_f32(const float* x, int64_t x_sample_stride, const float* mu, const float* rho, const float* s1, const float* s2,
                         int64_t param_stride, const float* eps, const float* bias, float* g, float* y_blocks, float* y, int64_t S,
                         int64_t B, int64_t D, int64_t G, int64_t n_out, int flags, whvi_stream_t stream)
{
    return stacked_fwd("stacked_fwd", 0, x, x_sample_stride, mu, rho, s1, s2, param_stride, eps, bias, g, y_blocks, y, S, B, D, G, n_out, flags, 0,
                       stream);
}

int whvi_stacked_fwd_bf16(const void* x, int64_t x_sample_stride, const float* mu, const float* rho, const float* s1, const float* s2,
                          int64_t param_stride, const float* eps, const float* bias, float* g, void* y_blocks, void* y, int64_t S,
                          int64_t B, int64_t D, int64_t G, int64_t n_out, int flags, whvi_stream_t stream)
{
    return stacked_fwd("stacked_fwd_bf16", 0, x, x_sample_stride, mu, rho, s1, s2, param_stride, eps, bias, g, y_blocks, y, S, B, D, G, n_out, flags,
                       1, stream);
}

int whvi_stacked_fwd_g_f32(const float* x, int64_t x_sample_stride, const float* g, const float* s1, const float* s2, int64_t param_stride,
                           const float* bias, float* y_blocks, float* y, int64_t S, int64_t B, int64_t D, int64_t G, int64_t n_out, int flags,
                           whvi_stream_t stream)
{
    return stacked_fwd("stacked_fwd_g", 1, x, x_sample_stride, nullptr, nullptr, s1, s2, param_stride, nullptr, bias, const_cast<float*>(g),
                       y_blocks, y, S, B, D, G, n_out, flags, 0, stream);
}

int whvi_stacked_fwd_g_bf16(const void* x, int64_t x_sample_stride, const float* g, const float* s1, const float* s2, int64_t param_stride,
                            const float* bias, void* y_blocks, void* y, int64_t S, int64_t B, int64_t D, int64_t G, int64_t n_out, int flags,
                            whvi_stream_t stream)
{
    return stacked_fwd("stacked_fwd_g_bf16", 1, x, x_sample_stride, nullptr, nullptr, s1, s2, param_stride, nullptr, bias, const_cast<float*>(g),
                       y_blocks, y, S, B, D, G, n_out, flags, 1, stream);
}

static size_t stacked_bwd_layout(int64_t S, int64_t B, int64_t D, int64_t G, int want_dx, size_t layer_ws, size_t* off_dx, size_t* off_dg,
                                 size_t* off_ws)
{
    const size_t blocks = sizeof(float) * size_t(G) * S * B * D;
    size_t o = blocks;                       // [0, blocks): dy in the block layout
    *off_dx = o;
    if (want_dx) o += blocks;
    *off_dg = o;
    o += sizeof(float) * size_t(G) * S * D;
    o = (o + 255) / 256 * 256;
    *off_ws = o;
    return o + layer_ws;
}

int whvi_stacked_bwd_workspace_bytes(int64_t S, int64_t B, int64_t D, int64_t G, int want_dx, size_t* bytes)
{
    if (!bytes) return fail(WHVI_E_NULL, "stacked_bwd_workspace_bytes: null pointer");
    if (int rc = check_stacked("stacked_bwd_workspace_bytes", S, B, D, G, G * D, 0, D)) return rc;
    *bytes = 0;
    if (S == 0 || B == 0) return WHVI_OK;
    size_t layer_ws = 0;
    LayerBwdCall c{};
    c.S = S * G;
    c.B = B;
    c.need_only = &layer_ws;
    if (int rc = launch_layer_bwd(c, D, nullptr)) return rc;
    size_t a, b, d;
    *bytes = stacked_bwd_layout(S, B, D, G, want_dx, layer_ws, &a, &b, &d);
    return WHVI_OK;
}

static int stacked_bwd_plan(const char* who, int64_t S, int64_t B, int64_t D, int64_t G, int want_dx, const void* workspace,
                            size_t workspace_bytes, size_t* layer_ws, size_t* off_dx, size_t* off_dg, size_t* off_ws)
{
    *layer_ws = 0;
    LayerBwdCall q{};
    q.S = S * G;
    q.B = B;
    q.need_only = layer_ws;
    if (int rc = launch_layer_bwd(q, D, nullptr)) return rc;
    const size_t need = stacked_bwd_layout(S, B, D, G, want_dx, *layer_ws, off_dx, off_dg, off_ws);
    if (!workspace || workspace_bytes < need) return fail(WHVI_E_WORKSPACE, "%s: workspace of %zu bytes needed, %zu given", who, need, workspace_bytes);
    return WHVI_OK;
}

// the layer's backward from dy (S, B, n_out) down to dg (G, S, D) and the per-block dx (left in the workspace for the caller's
// block sum); validated and planned by the callers.  bf16: dy is split into the first half of the (fp32-sized) dy-block region,
// and the per-block dx stay fp32 (summed and rounded once by stack_sum)
static int stacked_bwd_g(const float* x, int64_t xs, const float* dy, const float* g, const float* s1, const float* s2, int64_t param_stride,
                         float* dx, float* dg, float* ds1, float* ds2, float* dbias, void* workspace, size_t layer_ws, size_t off_dx,
                         size_t off_ws, int64_t S, int64_t B, int64_t D, int64_t G, int64_t n_out, int flags, cudaStream_t st, int bf16 = 0)
{
    char* base = static_cast<char*>(workspace);
    float* dyb = reinterpret_cast<float*>(base);
    float* dxb = dx ? reinterpret_cast<float*>(base + off_dx) : nullptr;
    if (int rc = launch_stack_split(dy, dyb, S * B, D, G, n_out, st, bf16)) return rc;
    LayerBwdCall c{x, dyb, g, s1, s2, nullptr, nullptr, nullptr, dxb, dg, ds1, ds2, dbias, reinterpret_cast<float*>(base + off_ws),
                   layer_ws, xs, S * G, B, flags & WHVI_LAYER_RELU_IN, nullptr};
    c.groups = G;
    c.pstride = param_stride;
    c.bf16 = bf16;
    c.dx_f32 = bf16;
    return launch_layer_bwd(c, D, st);
}

// a Stacked backward: down to (dmu, drho) through the diagonal reparameterisation, or -- from_g -- to dg (G, S, D) in the caller's
// buffer g_out (then rho, eps, dmu and drho are unused)
static int stacked_bwd(const char* who, int from_g, float* g_out, const void* x, int64_t x_sample_stride, const void* dy, const float* g, const float* rho,
                       const float* s1, const float* s2, int64_t param_stride, const float* eps, void* dx, int64_t n_in, float* dmu, float* drho,
                       float* ds1, float* ds2, float* dbias, void* workspace, size_t workspace_bytes, int64_t S, int64_t B, int64_t D, int64_t G,
                       int64_t n_out, int flags, int bf16, whvi_stream_t stream)
{
    if (int rc = check_stacked(who, S, B, D, G, n_out, x_sample_stride, param_stride)) return rc;
    if (flags & ~WHVI_LAYER_RELU_IN) return fail(WHVI_E_MODE, "%s: unknown flags %d", who, flags);
    if (dx && (n_in < 1 || n_in > D)) return fail(WHVI_E_SHAPE, "%s: n_in=%lld outside [1, D]", who, (long long)n_in);
    if ((from_g ? !g_out : (!dmu || !drho)) || !ds1 || !ds2) return fail(WHVI_E_NULL, "%s: null output pointer", who);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (S == 0 || B == 0) {
        if (from_g && S > 0) cudaMemsetAsync(g_out, 0, sizeof(float) * size_t(G) * S * D, st);
        for (float* p : {dmu, drho, ds1, ds2, dbias})
            if (p) cudaMemsetAsync(p, 0, sizeof(float) * size_t(G) * D, st);
        return check_launch(from_g ? "stacked_bwd_g(empty)" : "stacked_bwd(empty)");
    }
    if (!x || !dy || !g || (!from_g && (!rho || !eps)) || !s1 || !s2) return fail(WHVI_E_NULL, "%s: null pointer", who);
    if (!aligned16(x) || !aligned16(g) || !aligned16(s1) || !aligned16(s2) || !aligned16(g_out) || !aligned16(workspace))
        return fail(WHVI_E_ALIGN, "%s: pointers must be 16-byte aligned", who);
    if (bf16 && (B * D) % 8 != 0)   // the padded x and the block-layout dy reach the backward kernel by bulk copy (check_bf16_io)
        return fail(WHVI_E_SHAPE, "%s: B * D = %lld must be a multiple of 8 for bf16 activations (pad B)", who, (long long)(B * D));
    if (bf16 && (odd(dy) || odd(dx))) return fail(WHVI_E_ALIGN, "%s: dy and dx must be 2-byte aligned", who);
    size_t off_dx, off_dg, off_ws, layer_ws;
    if (int rc = stacked_bwd_plan(who, S, B, D, G, dx != nullptr, workspace, workspace_bytes, &layer_ws, &off_dx, &off_dg, &off_ws)) return rc;
    float* dg = from_g ? g_out : reinterpret_cast<float*>(static_cast<char*>(workspace) + off_dg);
    if (int rc = stacked_bwd_g(static_cast<const float*>(x), x_sample_stride, static_cast<const float*>(dy), g, s1, s2, param_stride,
                               static_cast<float*>(dx), dg, ds1, ds2, dbias, workspace, layer_ws, off_dx, off_ws, S, B, D, G, n_out, flags, st, bf16))
        return rc;
    if (!from_g)
        if (int rc = launch_reparam_diag_bwd(rho, eps, dg, dmu, drho, S, D, 0, st, G, param_stride)) return rc;
    if (dx)
        return launch_stack_sum(reinterpret_cast<float*>(static_cast<char*>(workspace) + off_dx), static_cast<float*>(dx), S * B, D, G, n_in, st, bf16);
    return WHVI_OK;
}

int whvi_stacked_bwd_f32(const float* x, int64_t x_sample_stride, const float* dy, const float* g, const float* rho, const float* s1,
                         const float* s2, int64_t param_stride, const float* eps, float* dx, int64_t n_in, float* dmu, float* drho,
                         float* ds1, float* ds2, float* dbias, void* workspace, size_t workspace_bytes, int64_t S, int64_t B, int64_t D,
                         int64_t G, int64_t n_out, int flags, whvi_stream_t stream)
{
    return stacked_bwd("stacked_bwd", 0, nullptr, x, x_sample_stride, dy, g, rho, s1, s2, param_stride, eps, dx, n_in, dmu, drho, ds1, ds2, dbias,
                       workspace, workspace_bytes, S, B, D, G, n_out, flags, 0, stream);
}

int whvi_stacked_bwd_bf16(const void* x, int64_t x_sample_stride, const void* dy, const float* g, const float* rho, const float* s1,
                          const float* s2, int64_t param_stride, const float* eps, void* dx, int64_t n_in, float* dmu, float* drho,
                          float* ds1, float* ds2, float* dbias, void* workspace, size_t workspace_bytes, int64_t S, int64_t B, int64_t D,
                          int64_t G, int64_t n_out, int flags, whvi_stream_t stream)
{
    return stacked_bwd("stacked_bwd_bf16", 0, nullptr, x, x_sample_stride, dy, g, rho, s1, s2, param_stride, eps, dx, n_in, dmu, drho, ds1, ds2, dbias,
                       workspace, workspace_bytes, S, B, D, G, n_out, flags, 1, stream);
}

int whvi_stacked_bwd_g_f32(const float* x, int64_t x_sample_stride, const float* dy, const float* g, const float* s1, const float* s2,
                           int64_t param_stride, float* dx, int64_t n_in, float* dg, float* ds1, float* ds2, float* dbias, void* workspace,
                           size_t workspace_bytes, int64_t S, int64_t B, int64_t D, int64_t G, int64_t n_out, int flags, whvi_stream_t stream)
{
    return stacked_bwd("stacked_bwd_g", 1, dg, x, x_sample_stride, dy, g, nullptr, s1, s2, param_stride, nullptr, dx, n_in, nullptr, nullptr, ds1,
                       ds2, dbias, workspace, workspace_bytes, S, B, D, G, n_out, flags, 0, stream);
}

int whvi_stacked_bwd_g_bf16(const void* x, int64_t x_sample_stride, const void* dy, const float* g, const float* s1, const float* s2,
                            int64_t param_stride, void* dx, int64_t n_in, float* dg, float* ds1, float* ds2, float* dbias, void* workspace,
                            size_t workspace_bytes, int64_t S, int64_t B, int64_t D, int64_t G, int64_t n_out, int flags, whvi_stream_t stream)
{
    return stacked_bwd("stacked_bwd_g_bf16", 1, dg, x, x_sample_stride, dy, g, nullptr, s1, s2, param_stride, nullptr, dx, n_in, nullptr, nullptr,
                       ds1, ds2, dbias, workspace, workspace_bytes, S, B, D, G, n_out, flags, 1, stream);
}
int whvi_kl_grouped_f32(const float* mu, const float* rho, float lambda_, int64_t D, int64_t G, int64_t param_stride, int mode,
                        float* out_kl, float* dmu, float* drho, float grad_scale, whvi_stream_t stream)
{
    if (D < 1 || G < 1 || (G > 1 && param_stride < D)) return fail(WHVI_E_SHAPE, "kl_grouped: D=%lld G=%lld stride=%lld", (long long)D, (long long)G, (long long)param_stride);
    if (mode != WHVI_KL_REFERENCE && mode != WHVI_KL_CONSISTENT) return fail(WHVI_E_MODE, "kl_grouped: unknown mode %d", mode);
    if (!(lambda_ > 0.f)) return fail(WHVI_E_SHAPE, "kl_grouped: lambda must be positive");
    if (!mu || !rho || !out_kl) return fail(WHVI_E_NULL, "kl_grouped: null pointer");
    if ((dmu == nullptr) != (drho == nullptr)) return fail(WHVI_E_NULL, "kl_grouped: dmu and drho must both be given or both NULL");
    return launch_kl(mu, rho, lambda_, D, mode, out_kl, dmu, drho, grad_scale, 0, static_cast<cudaStream_t>(stream), G, param_stride);
}

// ---- WHVIColumnMatrix as one call per direction (csrc/column.cu) --------------------------------------------------------
static int check_column(const char* who, int64_t S, int64_t B, int64_t D, int64_t n, int64_t xs, int transposed)
{
    if (S < 0 || B < 0 || D < 1 || !is_pow2(D) || D > (int64_t(1) << kMaxLog2D) || n < 1 || n > D || (D > 1 && n <= D / 2))
        return fail(WHVI_E_SHAPE, "%s: S=%lld B=%lld D=%lld n=%lld (D = next_pow2(n) <= 32768)", who, (long long)S, (long long)B, (long long)D, (long long)n);
    const int64_t row = transposed ? n : 1;
    if (xs != 0 && xs != B * row) return fail(WHVI_E_SHAPE, "%s: x_sample_stride must be 0 or B * %lld", who, (long long)row);
    return WHVI_OK;
}

// a Column forward: from (mu, rho, eps) drawn here into g, or -- from_g -- from g given (then mu, rho, eps are unused).  bf16: x and
// the plain form's y are bf16; the transposed form's y (S, B, 1) stays fp32
static int column_fwd(const char* who, int from_g, const void* x, int64_t x_sample_stride, const float* mu, const float* rho, const float* s1,
                      const float* s2, const float* eps, const float* bias, float* g, float* hg, void* y, int64_t S, int64_t B, int64_t D, int64_t n,
                      int transposed, int flags, int bf16, whvi_stream_t stream)
{
    if (int rc = check_column(who, S, B, D, n, x_sample_stride, transposed)) return rc;
    if (flags & ~WHVI_LAYER_RELU_OUT) return fail(WHVI_E_MODE, "%s: unknown flags %d", who, flags);
    if ((flags & WHVI_LAYER_RELU_OUT) && transposed) return fail(WHVI_E_MODE, "%s: RELU_OUT applies to the (.., 1) -> (.., n) form only", who);
    if (S == 0 || B == 0) return WHVI_OK;
    if (!x || (!from_g && (!mu || !rho || !eps)) || !s1 || !s2 || !g || !hg || !y) return fail(WHVI_E_NULL, "%s: null pointer", who);
    if (!aligned16(g) || !aligned16(hg)) return fail(WHVI_E_ALIGN, "%s: g and hg must be 16-byte aligned", who);
    if (bf16 && (odd(x) || (!transposed && odd(y)))) return fail(WHVI_E_ALIGN, "%s: bf16 pointers must be 2-byte aligned", who);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (from_g)
        return launch_column_fwd_g(static_cast<const float*>(x), x_sample_stride, g, s1, s2, bias, hg, static_cast<float*>(y), S, B, D, n,
                                   transposed, flags & WHVI_LAYER_RELU_OUT, st, bf16);
    return launch_column_fwd(static_cast<const float*>(x), x_sample_stride, mu, rho, s1, s2, eps, bias, g, hg, static_cast<float*>(y), S, B, D, n,
                             transposed, flags & WHVI_LAYER_RELU_OUT, st, bf16);
}

int whvi_column_fwd_f32(const float* x, int64_t x_sample_stride, const float* mu, const float* rho, const float* s1, const float* s2,
                        const float* eps, const float* bias, float* g, float* hg, float* y, int64_t S, int64_t B, int64_t D, int64_t n,
                        int transposed, int flags, whvi_stream_t stream)
{
    return column_fwd("column_fwd", 0, x, x_sample_stride, mu, rho, s1, s2, eps, bias, g, hg, y, S, B, D, n, transposed, flags, 0, stream);
}

int whvi_column_fwd_bf16(const void* x, int64_t x_sample_stride, const float* mu, const float* rho, const float* s1, const float* s2,
                         const float* eps, const float* bias, float* g, float* hg, void* y, int64_t S, int64_t B, int64_t D, int64_t n,
                         int transposed, int flags, whvi_stream_t stream)
{
    return column_fwd("column_fwd_bf16", 0, x, x_sample_stride, mu, rho, s1, s2, eps, bias, g, hg, y, S, B, D, n, transposed, flags, 1, stream);
}

int whvi_column_fwd_g_f32(const float* x, int64_t x_sample_stride, const float* g, const float* s1, const float* s2, const float* bias, float* hg,
                          float* y, int64_t S, int64_t B, int64_t D, int64_t n, int transposed, int flags, whvi_stream_t stream)
{
    return column_fwd("column_fwd_g", 1, x, x_sample_stride, nullptr, nullptr, s1, s2, nullptr, bias, const_cast<float*>(g), hg, y, S, B, D, n,
                      transposed, flags, 0, stream);
}

int whvi_column_fwd_g_bf16(const void* x, int64_t x_sample_stride, const float* g, const float* s1, const float* s2, const float* bias, float* hg,
                           void* y, int64_t S, int64_t B, int64_t D, int64_t n, int transposed, int flags, whvi_stream_t stream)
{
    return column_fwd("column_fwd_g_bf16", 1, x, x_sample_stride, nullptr, nullptr, s1, s2, nullptr, bias, const_cast<float*>(g), hg, y, S, B, D, n,
                      transposed, flags, 1, stream);
}

int whvi_column_bwd_workspace_bytes(int64_t S, int64_t D, int64_t n, size_t* bytes)
{
    if (!bytes) return fail(WHVI_E_NULL, "column_bwd_workspace_bytes: null pointer");
    if (S < 0 || D < 1 || n < 1 || n > D) return fail(WHVI_E_SHAPE, "column_bwd_workspace_bytes: S=%lld D=%lld n=%lld", (long long)S, (long long)D, (long long)n);
    *bytes = column_bwd_workspace_bytes(S, D, n);
    return WHVI_OK;
}

// a Column backward: down to (dmu, drho) through the diagonal reparameterisation, or -- from_g -- to dg (S, D) (then rho, eps, dmu and
// drho are unused).  bf16: x, dx and the plain form's dy are bf16; the transposed form's dy (S, B, 1) stays fp32
static int column_bwd(const char* who, int from_g, const void* x, int64_t x_sample_stride, const void* dy, const float* hg, const float* rho,
                      const float* s1, const float* s2, const float* eps, void* dx, float* dg, float* dmu, float* drho, float* ds1, float* ds2,
                      float* dbias, void* workspace, size_t workspace_bytes, int64_t S, int64_t B, int64_t D, int64_t n, int transposed, int flags,
                      int bf16, whvi_stream_t stream)
{
    if (int rc = check_column(who, S, B, D, n, x_sample_stride, transposed)) return rc;
    if (flags & ~WHVI_LAYER_RELU_IN) return fail(WHVI_E_MODE, "%s: unknown flags %d", who, flags);
    if ((flags & WHVI_LAYER_RELU_IN) && !transposed) return fail(WHVI_E_MODE, "%s: RELU_IN applies to the (.., n) -> (.., 1) form only", who);
    if ((from_g ? !dg : (!dmu || !drho)) || !ds1 || !ds2) return fail(WHVI_E_NULL, "%s: null output pointer", who);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (S == 0 || B == 0) {
        if (from_g && S > 0) cudaMemsetAsync(dg, 0, sizeof(float) * size_t(S) * D, st);
        for (float* p : {dmu, drho, ds1, ds2})
            if (p) cudaMemsetAsync(p, 0, sizeof(float) * size_t(D), st);
        if (dbias) cudaMemsetAsync(dbias, 0, sizeof(float) * size_t(transposed ? 1 : n), st);
        return check_launch(from_g ? "column_bwd_g(empty)" : "column_bwd(empty)");
    }
    if (!x || !dy || !hg || (!from_g && (!rho || !eps)) || !s1 || !s2) return fail(WHVI_E_NULL, "%s: null pointer", who);
    if (from_g ? !aligned16(workspace) || !aligned16(dg) : !aligned16(workspace))
        return fail(WHVI_E_ALIGN, from_g ? "%s: workspace and dg must be 16-byte aligned" : "%s: workspace must be 16-byte aligned", who);
    if (bf16 && (odd(x) || odd(dx) || (!transposed && odd(dy)))) return fail(WHVI_E_ALIGN, "%s: bf16 pointers must be 2-byte aligned", who);
    const size_t need = column_bwd_workspace_bytes(S, D, n);
    if (!workspace || workspace_bytes < need) return fail(WHVI_E_WORKSPACE, "%s: workspace of %zu bytes needed, %zu given", who, need, workspace_bytes);
    if (from_g)
        return launch_column_bwd_g(static_cast<const float*>(x), x_sample_stride, static_cast<const float*>(dy), hg, s1, s2, static_cast<float*>(dx),
                                   dg, ds1, ds2, dbias, static_cast<float*>(workspace), S, B, D, n, transposed, flags & WHVI_LAYER_RELU_IN, st, bf16);
    return launch_column_bwd(static_cast<const float*>(x), x_sample_stride, static_cast<const float*>(dy), hg, rho, s1, s2, eps, static_cast<float*>(dx),
                             dmu, drho, ds1, ds2, dbias, static_cast<float*>(workspace), S, B, D, n, transposed, flags & WHVI_LAYER_RELU_IN, st, bf16);
}

int whvi_column_bwd_f32(const float* x, int64_t x_sample_stride, const float* dy, const float* hg, const float* rho, const float* s1,
                        const float* s2, const float* eps, float* dx, float* dmu, float* drho, float* ds1, float* ds2, float* dbias,
                        void* workspace, size_t workspace_bytes, int64_t S, int64_t B, int64_t D, int64_t n, int transposed, int flags,
                        whvi_stream_t stream)
{
    return column_bwd("column_bwd", 0, x, x_sample_stride, dy, hg, rho, s1, s2, eps, dx, nullptr, dmu, drho, ds1, ds2, dbias, workspace,
                      workspace_bytes, S, B, D, n, transposed, flags, 0, stream);
}

int whvi_column_bwd_bf16(const void* x, int64_t x_sample_stride, const void* dy, const float* hg, const float* rho, const float* s1,
                         const float* s2, const float* eps, void* dx, float* dmu, float* drho, float* ds1, float* ds2, float* dbias,
                         void* workspace, size_t workspace_bytes, int64_t S, int64_t B, int64_t D, int64_t n, int transposed, int flags,
                         whvi_stream_t stream)
{
    return column_bwd("column_bwd_bf16", 0, x, x_sample_stride, dy, hg, rho, s1, s2, eps, dx, nullptr, dmu, drho, ds1, ds2, dbias, workspace,
                      workspace_bytes, S, B, D, n, transposed, flags, 1, stream);
}

int whvi_column_bwd_g_f32(const float* x, int64_t x_sample_stride, const float* dy, const float* hg, const float* s1, const float* s2, float* dx,
                          float* dg, float* ds1, float* ds2, float* dbias, void* workspace, size_t workspace_bytes, int64_t S, int64_t B, int64_t D,
                          int64_t n, int transposed, int flags, whvi_stream_t stream)
{
    return column_bwd("column_bwd_g", 1, x, x_sample_stride, dy, hg, nullptr, s1, s2, nullptr, dx, dg, nullptr, nullptr, ds1, ds2, dbias, workspace,
                      workspace_bytes, S, B, D, n, transposed, flags, 0, stream);
}

int whvi_column_bwd_g_bf16(const void* x, int64_t x_sample_stride, const void* dy, const float* hg, const float* s1, const float* s2, void* dx,
                           float* dg, float* ds1, float* ds2, float* dbias, void* workspace, size_t workspace_bytes, int64_t S, int64_t B, int64_t D,
                           int64_t n, int transposed, int flags, whvi_stream_t stream)
{
    return column_bwd("column_bwd_g_bf16", 1, x, x_sample_stride, dy, hg, nullptr, s1, s2, nullptr, dx, dg, nullptr, nullptr, ds1, ds2, dbias,
                      workspace, workspace_bytes, S, B, D, n, transposed, flags, 1, stream);
}

int whvi_layer_moments_f32(const float* x, int64_t x_sample_stride, const float* g, const float* s1, const float* s2,
                           const float* bias, float* sum_y, float* sum_y2, int64_t S, int64_t B, int64_t D, int flags,
                           whvi_stream_t stream)
{
    return whvi_layer_moments_add_f32(x, x_sample_stride, g, s1, s2, bias, nullptr, nullptr, sum_y, sum_y2, S, B, D, flags, stream);
}

int whvi_layer_moments_add_f32(const float* x, int64_t x_sample_stride, const float* g, const float* s1, const float* s2,
                               const float* bias, const float* in_sum_y, const float* in_sum_y2, float* sum_y, float* sum_y2,
                               int64_t S, int64_t B, int64_t D, int flags, whvi_stream_t stream)
{
    if (int rc = check_layer_shape("layer_moments", S, B, D, x_sample_stride, 32768)) return rc;
    if (D < 8192) return fail(WHVI_E_SHAPE, "layer_moments: D = %lld outside [8192, 32768] (use whvi_layer_fwd_fused_f32 + whvi_mc_moments_f32)", (long long)D);
    if (flags & ~(WHVI_LAYER_FROM_T2 | WHVI_LAYER_ACCUMULATE | 0xFF00)) return fail(WHVI_E_MODE, "layer_moments: unknown flags %d", flags);
    if ((flags & WHVI_LAYER_FROM_T2) && x_sample_stride != 0) return fail(WHVI_E_MODE, "layer_moments: FROM_T2 needs a shared (B, D) input");
    if (B == 0) return WHVI_OK;
    if (!x || !s1 || !s2 || !sum_y || (S > 0 && !g)) return fail(WHVI_E_NULL, "layer_moments: null pointer");
    if (!aligned16(x) || !aligned16(g) || !aligned16(s1) || !aligned16(s2) || !aligned16(bias) || !aligned16(sum_y) || !aligned16(sum_y2))
        return fail(WHVI_E_ALIGN, "layer_moments: pointers must be 16-byte aligned");
    if (!aligned16(in_sum_y) || !aligned16(in_sum_y2)) return fail(WHVI_E_ALIGN, "layer_moments: pointers must be 16-byte aligned");
    if (in_sum_y2 && !sum_y2) return fail(WHVI_E_NULL, "layer_moments: in_sum_y2 given without sum_y2");
    return launch_layer_moments(x, x_sample_stride, g, s1, s2, bias, sum_y, sum_y2, S, B, D, (flags & WHVI_LAYER_FROM_T2) ? 1 : 0,
                                (flags & WHVI_LAYER_ACCUMULATE) ? 1 : 0, (flags >> 8) & 0xFF, static_cast<cudaStream_t>(stream),
                                in_sum_y, in_sum_y2);
}

int whvi_adam_f32(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr,
                  const float* lr_dev, const float* step_dev, float beta1, float beta2, float eps, float grad_scale,
                  whvi_stream_t stream)
{
    if (n < 0) return fail(WHVI_E_SHAPE, "adam: n=%lld", (long long)n);
    if (n == 0) return WHVI_OK;
    if (!param || !grad || !exp_avg || !exp_avg_sq || !step_dev) return fail(WHVI_E_NULL, "adam: null pointer");
    if (!(beta1 >= 0.f && beta1 < 1.f && beta2 >= 0.f && beta2 < 1.f && eps >= 0.f))
        return fail(WHVI_E_MODE, "adam: betas must be in [0, 1) and eps >= 0");
    return launch_adam(param, grad, exp_avg, exp_avg_sq, n, lr, lr_dev, step_dev, beta1, beta2, eps, grad_scale,
                       static_cast<cudaStream_t>(stream));
}

int whvi_mc_moments_f32(const float* y, float* sum_y, float* sum_y2, int64_t S, int64_t n, int accumulate,
                        whvi_stream_t stream)
{
    if (S < 0 || n < 0 || (n & 3)) return fail(WHVI_E_SHAPE, "mc_moments: S=%lld n=%lld (n must be a multiple of 4)", (long long)S, (long long)n);
    if (n == 0) return WHVI_OK;
    if (!sum_y || (S > 0 && !y)) return fail(WHVI_E_NULL, "mc_moments: null pointer");
    if (!aligned16(y) || !aligned16(sum_y) || !aligned16(sum_y2)) return fail(WHVI_E_ALIGN, "mc_moments: pointers must be 16-byte aligned");
    return launch_mc_moments(y, n, accumulate ? sum_y : nullptr, accumulate ? sum_y2 : nullptr, sum_y, sum_y2, S, n,
                             static_cast<cudaStream_t>(stream));
}

int whvi_mc_moments_strided_f32(const float* y, int64_t y_sample_stride, const float* in_sum_y, const float* in_sum_y2,
                                float* out_sum_y, float* out_sum_y2, int64_t S, int64_t n, whvi_stream_t stream)
{
    if (S < 0 || n < 0 || (n & 3) || (y_sample_stride & 3) || y_sample_stride < n)
        return fail(WHVI_E_SHAPE, "mc_moments_strided: S=%lld n=%lld stride=%lld (n, stride multiples of 4, stride >= n)",
                    (long long)S, (long long)n, (long long)y_sample_stride);
    if (n == 0) return WHVI_OK;
    if (!out_sum_y || (S > 0 && !y)) return fail(WHVI_E_NULL, "mc_moments_strided: null pointer");
    if (!aligned16(y) || !aligned16(in_sum_y) || !aligned16(in_sum_y2) || !aligned16(out_sum_y) || !aligned16(out_sum_y2))
        return fail(WHVI_E_ALIGN, "mc_moments_strided: pointers must be 16-byte aligned");
    return launch_mc_moments(y, y_sample_stride, in_sum_y, in_sum_y2, out_sum_y, out_sum_y2, S, n, static_cast<cudaStream_t>(stream));
}

// ---- categorical likelihood (csrc/categorical.cu) -----------------------------------------------------------------------
static bool aligned(const void* p, uintptr_t bytes) { return (reinterpret_cast<uintptr_t>(p) & (bytes - 1)) == 0; }

static int check_categorical(const char* who, int64_t S, int64_t B, int64_t K)
{
    if (S < 0 || B < 0) return fail(WHVI_E_SHAPE, "%s: S=%lld B=%lld", who, (long long)S, (long long)B);
    if (K < 2 || K > 65536) return fail(WHVI_E_SHAPE, "%s: K = %lld outside [2, 65536]", who, (long long)K);
    if (B > (int64_t(1) << 46) || (S > 0 && B > (int64_t(1) << 46) / S)) return fail(WHVI_E_SHAPE, "%s: S * B too large", who);
    return WHVI_OK;
}

int whvi_categorical_sizes(int64_t R, int64_t K, size_t* workspace_bytes)
{
    if (!workspace_bytes) return fail(WHVI_E_NULL, "categorical_sizes: null pointer");
    if (int rc = check_categorical("categorical_sizes", R, 1, K)) return rc;
    *workspace_bytes = categorical_workspace_bytes(R, K);
    return WHVI_OK;
}

static int categorical_nll(const char* who, const void* logits, size_t elem, const int64_t* labels, float* lse, float* total, void* workspace,
                           size_t workspace_bytes, int64_t S, int64_t B, int64_t K, whvi_stream_t stream)
{
    if (int rc = check_categorical(who, S, B, K)) return rc;
    if (!total || (S * B > 0 && (!logits || !labels))) return fail(WHVI_E_NULL, "%s: null pointer", who);
    if (!aligned(logits, elem) || !aligned(labels, 8) || !aligned(lse, 4) || !aligned(total, 4))
        return fail(WHVI_E_ALIGN, "%s: logits, labels, lse and total must be aligned to their element size", who);
    const size_t need = categorical_workspace_bytes(S * B, K);
    if (!workspace || workspace_bytes < need || !aligned(workspace, 8))
        return fail(WHVI_E_WORKSPACE, "%s: workspace of %zu bytes (8-byte aligned) needed, %zu given", who, need, workspace_bytes);
    return launch_categorical_nll(logits, labels, lse, total, workspace, S, B, K, elem == 2, static_cast<cudaStream_t>(stream));
}

int whvi_categorical_nll_f32(const float* logits, const int64_t* labels, float* lse, float* total, void* workspace, size_t workspace_bytes,
                             int64_t S, int64_t B, int64_t K, whvi_stream_t stream)
{
    return categorical_nll("categorical_nll_f32", logits, 4, labels, lse, total, workspace, workspace_bytes, S, B, K, stream);
}

int whvi_categorical_nll_bf16(const void* logits, const int64_t* labels, float* lse, float* total, void* workspace, size_t workspace_bytes,
                              int64_t S, int64_t B, int64_t K, whvi_stream_t stream)
{
    return categorical_nll("categorical_nll_bf16", logits, 2, labels, lse, total, workspace, workspace_bytes, S, B, K, stream);
}

static int categorical_nll_bwd(const char* who, const void* logits, size_t elem, const int64_t* labels, const float* lse, const float* c,
                               void* dz, int64_t S, int64_t B, int64_t K, whvi_stream_t stream)
{
    if (int rc = check_categorical(who, S, B, K)) return rc;
    if (S * B == 0) return WHVI_OK;
    if (!logits || !labels || !lse || !dz) return fail(WHVI_E_NULL, "%s: null pointer", who);
    if (!aligned(logits, elem) || !aligned(dz, elem) || !aligned(labels, 8) || !aligned(lse, 4) || !aligned(c, 4))
        return fail(WHVI_E_ALIGN, "%s: logits, dz, labels, lse and c must be aligned to their element size", who);
    return launch_categorical_nll_bwd(logits, labels, lse, c, dz, S, B, K, elem == 2, static_cast<cudaStream_t>(stream));
}

int whvi_categorical_nll_bwd_f32(const float* logits, const int64_t* labels, const float* lse, const float* c, float* dz, int64_t S,
                                 int64_t B, int64_t K, whvi_stream_t stream)
{
    return categorical_nll_bwd("categorical_nll_bwd_f32", logits, 4, labels, lse, c, dz, S, B, K, stream);
}

int whvi_categorical_nll_bwd_bf16(const void* logits, const int64_t* labels, const float* lse, const float* c, void* dz, int64_t S,
                                  int64_t B, int64_t K, whvi_stream_t stream)
{
    return categorical_nll_bwd("categorical_nll_bwd_bf16", logits, 2, labels, lse, c, dz, S, B, K, stream);
}

static int categorical_predictive(const char* who, const void* logits, size_t elem, int64_t sample_stride, const int64_t* labels,
                                  float* prob_sum, float* loglik_sum, int64_t S, int64_t B, int64_t K, int flags, whvi_stream_t stream)
{
    if (int rc = check_categorical(who, S, B, K)) return rc;
    if (flags & ~WHVI_CATEGORICAL_ACCUMULATE) return fail(WHVI_E_MODE, "%s: unknown flags %d", who, flags);
    if (S > 1 && sample_stride < B * K)
        return fail(WHVI_E_SHAPE, "%s: sample_stride=%lld below B * K = %lld", who, (long long)sample_stride, (long long)(B * K));
    if (S > 1 && sample_stride > (int64_t(1) << 62) / S) return fail(WHVI_E_SHAPE, "%s: sample_stride too large", who);
    if ((labels == nullptr) != (loglik_sum == nullptr)) return fail(WHVI_E_NULL, "%s: labels and loglik_sum must both be given or both NULL", who);
    if (B == 0) return WHVI_OK;
    if (!prob_sum || (S > 0 && !logits)) return fail(WHVI_E_NULL, "%s: null pointer", who);
    if (!aligned(logits, elem) || !aligned(labels, 8) || !aligned(prob_sum, 4) || !aligned(loglik_sum, 4))
        return fail(WHVI_E_ALIGN, "%s: logits, labels, prob_sum and loglik_sum must be aligned to their element size", who);
    return launch_categorical_predictive(logits, sample_stride, labels, prob_sum, loglik_sum, S, B, K, flags & WHVI_CATEGORICAL_ACCUMULATE,
                                         elem == 2, static_cast<cudaStream_t>(stream));
}

int whvi_categorical_predictive_f32(const float* logits, int64_t sample_stride, const int64_t* labels, float* prob_sum, float* loglik_sum,
                                    int64_t S, int64_t B, int64_t K, int flags, whvi_stream_t stream)
{
    return categorical_predictive("categorical_predictive_f32", logits, 4, sample_stride, labels, prob_sum, loglik_sum, S, B, K, flags, stream);
}

int whvi_categorical_predictive_bf16(const void* logits, int64_t sample_stride, const int64_t* labels, float* prob_sum, float* loglik_sum,
                                     int64_t S, int64_t B, int64_t K, int flags, whvi_stream_t stream)
{
    return categorical_predictive("categorical_predictive_bf16", logits, 2, sample_stride, labels, prob_sum, loglik_sum, S, B, K, flags,
                                  stream);
}

// ---- convolution patches (csrc/conv.cu) ---------------------------------------------------------------------------------
static int check_conv(const char* who, int64_t S, int64_t B, int64_t H, int64_t W, int64_t C, int64_t kh, int64_t kw, int64_t sh,
                      int64_t sw, int64_t ph, int64_t pw, int64_t dh, int64_t dw, int64_t ld, ConvGeom* g)
{
    constexpr int64_t kLim = int64_t(1) << 24;
    if (S < 0 || B < 0) return fail(WHVI_E_SHAPE, "%s: S=%lld B=%lld", who, (long long)S, (long long)B);
    const int64_t pos[] = {H, W, C, kh, kw, sh, sw, dh, dw};
    for (int64_t v : pos)
        if (v < 1 || v >= kLim) return fail(WHVI_E_SHAPE, "%s: H, W, C, kernel, stride and dilation must lie in [1, 2^24)", who);
    if (ph < 0 || pw < 0 || ph >= kLim || pw >= kLim) return fail(WHVI_E_SHAPE, "%s: padding must lie in [0, 2^24)", who);
    const int64_t ext_h = dh * (kh - 1) + 1, ext_w = dw * (kw - 1) + 1;
    if (ext_h >= kLim || ext_w >= kLim) return fail(WHVI_E_SHAPE, "%s: dilated kernel extent must be below 2^24", who);
    const int64_t num_h = H + 2 * ph - ext_h, num_w = W + 2 * pw - ext_w;
    if (num_h < 0 || num_w < 0)
        return fail(WHVI_E_SHAPE, "%s: the dilated kernel (%lld x %lld) exceeds the padded image (%lld x %lld): Ho or Wo <= 0", who,
                    (long long)ext_h, (long long)ext_w, (long long)(H + 2 * ph), (long long)(W + 2 * pw));
    const int64_t Ho = num_h / sh + 1, Wo = num_w / sw + 1;
    if (kh * kw > (int64_t(1) << 31) / C || ld > INT32_MAX)
        return fail(WHVI_E_SHAPE, "%s: C * kh * kw and ld must stay below 2^31", who);
    const int64_t n_in = C * kh * kw;
    if (ld < n_in) return fail(WHVI_E_SHAPE, "%s: ld=%lld below n_in = C * kh * kw = %lld", who, (long long)ld, (long long)n_in);
    // the larger side, S * B * max(Ho * Wo * ld, H * W * C) elements, must stay below 2^62 (Ho * Wo and H * W are below 2^52)
    constexpr int64_t kMaxElems = int64_t(1) << 62;
    if (Ho * Wo > kMaxElems / ld || H * W > kMaxElems / C) return fail(WHVI_E_SHAPE, "%s: too many elements", who);
    const int64_t per = Ho * Wo * ld > H * W * C ? Ho * Wo * ld : H * W * C;
    if ((B > 0 && S > kMaxElems / B) || (S * B > 0 && S * B > kMaxElems / per)) return fail(WHVI_E_SHAPE, "%s: too many elements", who);
    *g = ConvGeom{S, B, int(H), int(W), int(C), int(kh), int(kw), int(sh), int(sw), int(ph), int(pw), int(dh), int(dw), int(Ho), int(Wo)};
    return WHVI_OK;
}

static int im2col(const char* who, const void* x, int64_t x_sample_stride, void* patches, size_t elem, int64_t S, int64_t B, int64_t H,
                  int64_t W, int64_t C, int64_t kh, int64_t kw, int64_t sh, int64_t sw, int64_t ph, int64_t pw, int64_t dh, int64_t dw,
                  int64_t ld, whvi_stream_t stream)
{
    ConvGeom g;
    if (int rc = check_conv(who, S, B, H, W, C, kh, kw, sh, sw, ph, pw, dh, dw, ld, &g)) return rc;
    if (x_sample_stride != 0 && x_sample_stride != B * H * W * C)
        return fail(WHVI_E_SHAPE, "%s: x_sample_stride must be 0 or B*H*W*C", who);
    if (S * B == 0) return WHVI_OK;
    if (!x || !patches) return fail(WHVI_E_NULL, "%s: null pointer", who);
    if (!aligned(x, elem) || !aligned(patches, elem)) return fail(WHVI_E_ALIGN, "%s: x and patches must be aligned to their element size", who);
    return launch_im2col(x, x_sample_stride, patches, g, ld, elem == 2, static_cast<cudaStream_t>(stream));
}

int whvi_im2col_f32(const float* x, int64_t x_sample_stride, float* patches, int64_t S, int64_t B, int64_t H, int64_t W, int64_t C,
                    int64_t kh, int64_t kw, int64_t stride_h, int64_t stride_w, int64_t pad_h, int64_t pad_w, int64_t dil_h,
                    int64_t dil_w, int64_t ld, whvi_stream_t stream)
{
    return im2col("im2col_f32", x, x_sample_stride, patches, 4, S, B, H, W, C, kh, kw, stride_h, stride_w, pad_h, pad_w, dil_h, dil_w,
                  ld, stream);
}

int whvi_im2col_bf16(const void* x, int64_t x_sample_stride, void* patches, int64_t S, int64_t B, int64_t H, int64_t W, int64_t C,
                     int64_t kh, int64_t kw, int64_t stride_h, int64_t stride_w, int64_t pad_h, int64_t pad_w, int64_t dil_h,
                     int64_t dil_w, int64_t ld, whvi_stream_t stream)
{
    return im2col("im2col_bf16", x, x_sample_stride, patches, 2, S, B, H, W, C, kh, kw, stride_h, stride_w, pad_h, pad_w, dil_h, dil_w,
                  ld, stream);
}

static int col2im(const char* who, const void* dpatches, int64_t ld, void* dx, size_t elem, int64_t S, int64_t B, int64_t H, int64_t W,
                  int64_t C, int64_t kh, int64_t kw, int64_t sh, int64_t sw, int64_t ph, int64_t pw, int64_t dh, int64_t dw, int flags,
                  whvi_stream_t stream)
{
    ConvGeom g;
    if (int rc = check_conv(who, S, B, H, W, C, kh, kw, sh, sw, ph, pw, dh, dw, ld, &g)) return rc;
    if (flags & ~WHVI_COL2IM_SUM_SAMPLES) return fail(WHVI_E_MODE, "%s: unknown flags %d", who, flags);
    const int sum = flags & WHVI_COL2IM_SUM_SAMPLES;
    if ((sum ? 1 : S) * B == 0) return WHVI_OK;
    if (!dx || (S > 0 && !dpatches)) return fail(WHVI_E_NULL, "%s: null pointer", who);
    if (!aligned(dpatches, elem) || !aligned(dx, elem)) return fail(WHVI_E_ALIGN, "%s: dpatches and dx must be aligned to their element size", who);
    return launch_col2im(dpatches, ld, dx, g, sum, elem == 2, static_cast<cudaStream_t>(stream));
}

int whvi_col2im_f32(const float* dpatches, int64_t ld, float* dx, int64_t S, int64_t B, int64_t H, int64_t W, int64_t C, int64_t kh,
                    int64_t kw, int64_t stride_h, int64_t stride_w, int64_t pad_h, int64_t pad_w, int64_t dil_h, int64_t dil_w, int flags,
                    whvi_stream_t stream)
{
    return col2im("col2im_f32", dpatches, ld, dx, 4, S, B, H, W, C, kh, kw, stride_h, stride_w, pad_h, pad_w, dil_h, dil_w, flags, stream);
}

int whvi_col2im_bf16(const void* dpatches, int64_t ld, void* dx, int64_t S, int64_t B, int64_t H, int64_t W, int64_t C, int64_t kh,
                     int64_t kw, int64_t stride_h, int64_t stride_w, int64_t pad_h, int64_t pad_w, int64_t dil_h, int64_t dil_w, int flags,
                     whvi_stream_t stream)
{
    return col2im("col2im_bf16", dpatches, ld, dx, 2, S, B, H, W, C, kh, kw, stride_h, stride_w, pad_h, pad_w, dil_h, dil_w, flags, stream);
}

}  // extern "C"
