// Shared host-side plumbing of libwhvi_b200: status codes, thread-local error text,
// launch checks.  No torch headers anywhere in this library.
#pragma once
#include <cuda_runtime.h>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include "../../include/whvi_b200.h"

namespace whvi {

char* error_buffer();  // thread-local, 512 bytes (api.cu)

inline int fail(int code, const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(error_buffer(), 512, fmt, ap);
    va_end(ap);
    return code;
}

inline int check_launch(const char* what)
{
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(static_cast<int>(e), "%s: %s", what, cudaGetErrorString(e));
    return WHVI_OK;
}

inline bool is_pow2(int64_t v) { return v > 0 && (v & (v - 1)) == 0; }
inline int ilog2(int64_t v)
{
    int k = 0;
    while ((int64_t(1) << k) < v) ++k;
    return k;
}
inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// Opt a kernel in to > 48 KB of dynamic shared memory, once per (kernel, device).
template <class Kernel>
inline int ensure_smem(Kernel kernel, size_t bytes, unsigned char* done_flags /*[64]*/)
{
    if (bytes <= 40 * 1024) return WHVI_OK;  // static __shared__ of the kernel counts against the 48 KB default too
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 0 && dev < 64 && done_flags[dev]) return WHVI_OK;
    const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(bytes));
    if (e != cudaSuccess) return fail(static_cast<int>(e), "cudaFuncSetAttribute(smem=%zu): %s", bytes, cudaGetErrorString(e));
    if (dev >= 0 && dev < 64) done_flags[dev] = 1;
    return WHVI_OK;
}

constexpr int kMaxLog2D = 15;       // single-pass kernels keep a whole row in one CTA's shared memory
constexpr int kMaxLog2Dmulti = 30;  // multi-pass global variant beyond that

int launch_fwht(const float* in, float* out, int64_t rows, int64_t D, cudaStream_t stream);
int launch_fwht_scaled(const float* in, const float* scale, float* out, int64_t rows, int64_t D, cudaStream_t stream);
int launch_fwht_bf16(const void* in, void* out, int64_t rows, int64_t D, cudaStream_t stream);
int launch_fwht_f64(const double* in, double* out, int64_t rows, int64_t D, cudaStream_t stream);
struct LayerFwdCall {
    const float *x, *g, *s1, *s2, *bias, *target;
    float *y, *sq_partials;
    int64_t xs, S, B;
    int relu_out;
    size_t* partials_needed;  // query mode: number of floats of sq_partials
    int from_t2 = 0;          // x already holds H(s2 * x)
    // grouped launch (a Stacked layer's blocks as extra samples, src/weights.py:179-180): S counts VIRTUAL samples
    // s' = block * (S / groups) + sample; block k reads s1/s2 at + k * pstride floats, bias at + k * bstride, and the input
    // of sample s' % (S / groups)
    int64_t groups = 1, pstride = 0, bstride = 0;
    int bf16 = 0;             // x and y are bf16 in HBM (arithmetic stays fp32)
};
struct LayerBwdCall {
    const float *x, *dy, *g, *s1, *s2, *target, *coef, *dy_scale;
    float *dx, *dg, *ds1, *ds2, *dbias, *ws;
    size_t ws_bytes;
    int64_t xs, S, B;
    int relu_in;
    size_t* need_only;  // query mode: workspace bytes
    int64_t groups = 1, pstride = 0;  // grouped launch (see LayerFwdCall): ds1 / ds2 / dbias are (groups, D)
    int bf16 = 0;             // x, dy and dx are bf16 in HBM (behind the float pointers; arithmetic and workspace stay fp32)
    int dx_f32 = 0;           // with bf16: dx stays fp32 (the grouped backward's per-block dx, summed and rounded once by the caller)
};
struct LayerLossCall {  // fused last layer: forward + Gaussian-MNLL residual + backward in one pass
    const float *x, *g, *s1, *s2, *bias, *target;
    float *dx, *dg, *ds1, *ds2, *dbias, *sq_partials, *ws;
    size_t ws_bytes;
    int64_t xs, S, B;
    int relu_in;
    size_t* need_ws;      // query mode
    int64_t* need_sq;     // query mode
    int bf16 = 0;         // x and dx are bf16 in HBM (behind the float pointers); target, parameters and arithmetic stay fp32
};
int launch_layer_loss(const LayerLossCall& c, int64_t D, cudaStream_t stream);
int launch_bwd_reduce(float* ws, float* dg, float* ds1, float* ds2, float* dbias, int64_t S, int slabs_per_sample,
                      int64_t tile, int64_t D, cudaStream_t stream, int64_t groups = 1);
int launch_layer_fwd(const LayerFwdCall& c, int64_t D, cudaStream_t stream);
int launch_layer_bwd(const LayerBwdCall& c, int64_t D, cudaStream_t stream);
int launch_reparam_diag(const float* mu, const float* rho, const float* eps, float* g, int64_t S, int64_t D,
                        cudaStream_t stream, int64_t groups = 1, int64_t pstride = 0);
size_t reparam_dense_workspace_bytes(int64_t S, int64_t D);
int launch_reparam_dense(const float* mu, const float* L, const float* eps, float* g, int64_t S, int64_t D, float* ws, size_t ws_bytes,
                         cudaStream_t stream);
int launch_reparam_dense_bwd(const float* dgT, const float* eT, float* dL, int64_t Sp, int64_t D, cudaStream_t stream);
int launch_kl_dense(const float* mu, const float* L, float lambda_, int64_t D, float* out, float* dmu, float* dL, float grad_scale,
                    double* row_sq, cudaStream_t stream);
size_t reparam_dense_grouped_workspace_bytes(int64_t S, int64_t D);
int launch_reparam_dense_grouped(const float* mu, int64_t mu_stride, const float* L, int64_t L_stride, const float* eps, float* g, int64_t S,
                                 int64_t D, int64_t G, float* ws, size_t ws_bytes, cudaStream_t stream);
int launch_reparam_dense_grouped_bwd(const float* eps, const float* dg, float* dmu, float* dL, int64_t S, int64_t D, int64_t G, float* ws,
                                     size_t ws_bytes, cudaStream_t stream);
int launch_kl_dense_grouped(const float* mu, int64_t mu_stride, const float* L, int64_t L_stride, float lambda_, int64_t D, int64_t G, float* out,
                            float* dmu, float* dL, float grad_scale, double* row_sq, cudaStream_t stream);
// Column layer; bf16 != 0: x, dx and the plain form's y / dy are bf16 behind the float pointers (column.cu)
int launch_column_fwd_g(const float* x, int64_t xs, const float* g, const float* s1, const float* s2, const float* bias, float* hg, float* y,
                        int64_t S, int64_t B, int64_t D, int64_t n, int transposed, int relu_out, cudaStream_t st, int bf16 = 0);
int launch_column_bwd_g(const float* x, int64_t xs, const float* dy, const float* hg, const float* s1, const float* s2, float* dx, float* dg,
                        float* ds1, float* ds2, float* dbias, float* ws, int64_t S, int64_t B, int64_t D, int64_t n, int transposed, int relu_in,
                        cudaStream_t st, int bf16 = 0);
int launch_reparam_diag_bwd(const float* rho, const float* eps, const float* dg, float* dmu, float* drho, int64_t S,
                            int64_t D, int accumulate, cudaStream_t stream, int64_t groups = 1, int64_t pstride = 0);
// the Stacked interleave kernels; bf16 != 0: the activation side (in / out / dx) is bf16 behind the float pointers (the blocks of
// split and concat are bf16 too, stack_sum's dxb stays fp32 and its output is rounded once)
int launch_stack_split(const float* in, float* blocks, int64_t R, int64_t D, int64_t G, int64_t n_out, cudaStream_t stream, int bf16 = 0);
int launch_stack_concat(const float* blocks, float* out, int64_t R, int64_t D, int64_t G, int64_t n_out, cudaStream_t stream, int bf16 = 0);
int launch_stack_sum(const float* dxb, float* dx, int64_t R, int64_t D, int64_t G, int64_t n_in, cudaStream_t stream, int bf16 = 0);
int launch_column_fwd(const float* x, int64_t xs, const float* mu, const float* rho, const float* s1, const float* s2, const float* eps,
                      const float* bias, float* g, float* hg, float* y, int64_t S, int64_t B, int64_t D, int64_t n, int transposed, int relu_out,
                      cudaStream_t st, int bf16 = 0);
size_t column_bwd_workspace_bytes(int64_t S, int64_t D, int64_t n);
int launch_column_bwd(const float* x, int64_t xs, const float* dy, const float* hg, const float* rho, const float* s1, const float* s2,
                      const float* eps, float* dx, float* dmu, float* drho, float* ds1, float* ds2, float* dbias, float* ws, int64_t S,
                      int64_t B, int64_t D, int64_t n, int transposed, int relu_in, cudaStream_t st, int bf16 = 0);
int launch_layer_moments(const float* x, int64_t xs, const float* g, const float* s1, const float* s2, const float* bias, float* sum_y,
                         float* sum_y2, int64_t S, int64_t B, int64_t D, int from_t2, int accumulate, int reserve_sms, cudaStream_t stream,
                         const float* in_y = nullptr, const float* in_y2 = nullptr);
int launch_mc_moments(const float* y, int64_t y_sample_stride, const float* in_y, const float* in_y2, float* out_y, float* out_y2,
                      int64_t S, int64_t n, cudaStream_t stream);
int launch_adam(float* p, const float* g, float* m, float* v, int64_t n, float lr, const float* lr_dev, const float* step,
                float b1, float b2, float eps, float grad_scale, cudaStream_t stream);
int launch_kl(const float* mu, const float* rho, float lambda_, int64_t D, int mode, float* out, float* dmu, float* drho,
              float grad_scale, int accumulate, cudaStream_t stream, int64_t groups = 1, int64_t pstride = 0);
// categorical likelihood (categorical.cu); bf16 != 0: the logits and dz are bf16 behind the void pointers
size_t categorical_workspace_bytes(int64_t R, int64_t K);
// the _ex calls' options: on = false runs the plain instances (weight NULL, eps 0, no ignore_index)
struct CategoricalOpts {
    bool on;
    const float* weight;   // (K) or NULL for ones
    float eps;             // label smoothing in [0, 1]
    int64_t ignore_index;
    int ignore;            // rows with y_b == ignore_index add 0 and get a zero dz row
};
int launch_categorical_nll(const void* z, const int64_t* labels, float* lse, float* total, void* ws, int64_t S, int64_t B, int64_t K,
                           int bf16, const CategoricalOpts& o, cudaStream_t st);
int launch_categorical_nll_bwd(const void* z, const int64_t* labels, const float* lse, const float* c, void* dz, int64_t S, int64_t B,
                               int64_t K, int bf16, const CategoricalOpts& o, cudaStream_t st);
// ent_sum != NULL: the uncertainty sums as well (logpred with the labels, else NULL)
int launch_categorical_predictive(const void* z, int64_t sample_stride, const int64_t* labels, float* prob_sum, float* loglik_sum,
                                  float* logpred, float* ent_sum, int64_t S, int64_t B, int64_t K, int accumulate, int bf16,
                                  cudaStream_t st);
// patch gather / scatter of WHVIConv2d (conv.cu); validated geometry, every spatial quantity below 2^24
struct ConvGeom {
    int64_t S, B;
    int H, W, C, kh, kw, sh, sw, ph, pw, dh, dw, Ho, Wo;
};
int launch_im2col(const void* x, int64_t xs, void* out, const ConvGeom& g, int64_t ld, int bf16, cudaStream_t st);
int launch_col2im(const void* dp, int64_t ld, void* dx, const ConvGeom& g, int sum_samples, int bf16, cudaStream_t st);

}  // namespace whvi
