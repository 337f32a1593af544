// Categorical (softmax) likelihood of a WHVI classifier (not in the reference, whose networks only regress):
//   categorical_nll          lse_r = log sum_k exp(z_rk) (max-subtracted, online), loss_r = lse_r - z_{r, y_b},
//                            total = sum_r loss_r: fp64 per-CTA partials, then one CTA sums them in a fixed order
//   categorical_nll_bwd      dz_rk = c (exp(z_rk - lse_r) - [k = y_b]),  c a device scalar
//   categorical_predictive   prob_sum[b, :] (+)= sum_s softmax(z_{s,b}),  loglik_sum[b] (+)= sum_s log p_s(y_b),  s ascending
// Rows r = s * B + b of the (S, B, K) logits, labels (B) int64.
//
// Work split: a GROUP of TPR threads owns a row.  K <= 32: TPR = next_pow2(K), so a warp holds 32 / TPR rows; K <= 2048:
// a warp per row; beyond, a CTA per row.  Lane j of a group handles the elements k = j, j + TPR, ... in ascending order with
// an online (max, sum) pair, and the pairs are combined by a fixed butterfly (and, for a CTA, a fixed sweep over the warps).
// The loads are element-wise and coalesced across the group: the element-to-lane assignment depends on k alone, never on a
// row's address, so rows need no alignment and the bf16 instances -- the fp32 code on the widened logits -- give the fp32
// instances' results bit for bit.  Bandwidth-bound: the forward and the backward read each logit once (the backward also
// writes dz), the predictive reads each row twice per sample (the second pass from L1 / L2).
//
// A label outside [0, K) is never dereferenced: its row's loss, log p and dz row are NaN instead.
#include <cuda_bf16.h>

#include <type_traits>

#include "common.cuh"

namespace whvi {
namespace {

constexpr int kThreads = 256;
constexpr int64_t kMaxCtas = 148 * 16;

__device__ __forceinline__ float ldz(const float* p, int64_t i) { return __ldg(p + i); }
__device__ __forceinline__ float ldz(const __nv_bfloat16* p, int64_t i) { return __bfloat162float(p[i]); }
__device__ __forceinline__ void stz(float* p, int64_t i, float v) { p[i] = v; }
__device__ __forceinline__ void stz(__nv_bfloat16* p, int64_t i, float v) { p[i] = __float2bfloat16_rn(v); }

__device__ __forceinline__ float qnan() { return __int_as_float(0x7fc00000); }

// running max m and sum s of exp(z - m)
struct MaxSum {
    float m, s;
};

__device__ __forceinline__ void push(MaxSum& a, float z)
{
    if (z > a.m) {
        a.s = a.s * expf(a.m - z) + 1.f;
        a.m = z;
    } else {
        a.s += z == -INFINITY ? 0.f : expf(z - a.m);   // a masked class adds nothing (and -inf - -inf is no NaN)
    }
}

// symmetric in its arguments bit for bit, so every lane of a butterfly ends with the same pair
__device__ __forceinline__ MaxSum combine(MaxSum a, MaxSum b)
{
    const float m = fmaxf(a.m, b.m);
    return {m, (a.m == m ? a.s : a.s * expf(a.m - m)) + (b.m == m ? b.s : b.s * expf(b.m - m))};
}

// log sum_k exp(row[k]) in every thread of the group.  TPR == kThreads synchronises the CTA: call it CTA-uniformly.
template <int TPR, typename T>
__device__ __forceinline__ float row_lse(const T* row, int K, int lane, bool valid)
{
    MaxSum a{-INFINITY, 0.f};
    if (valid) {
#pragma unroll 4
        for (int k = lane; k < K; k += TPR) push(a, ldz(row, k));
    }
    constexpr int width = TPR < 32 ? TPR : 32;
#pragma unroll
    for (int o = width / 2; o > 0; o >>= 1)
        a = combine(a, MaxSum{__shfl_xor_sync(0xffffffffu, a.m, o), __shfl_xor_sync(0xffffffffu, a.s, o)});
    if constexpr (TPR > 32) {
        __shared__ MaxSum warps[TPR / 32];
        if ((threadIdx.x & 31) == 0) warps[threadIdx.x >> 5] = a;
        __syncthreads();
        a = warps[0];
#pragma unroll
        for (int w = 1; w < TPR / 32; ++w) a = combine(a, warps[w]);
        __syncthreads();   // the next row may overwrite warps[]
    }
    return a.m + logf(a.s);
}

template <int TPR, typename T>
__global__ void __launch_bounds__(kThreads)
categorical_nll_kernel(const T* __restrict__ z, const int64_t* __restrict__ labels, float* __restrict__ lse_out,
                       double* __restrict__ partials, int64_t R, int64_t B, int K)
{
    constexpr int G = kThreads / TPR;
    const int g = threadIdx.x / TPR, lane = threadIdx.x % TPR;
    double acc = 0.0;
    const int64_t blocks = (R + G - 1) / G;
    for (int64_t blk = blockIdx.x; blk < blocks; blk += gridDim.x) {   // CTA-uniform trip count
        const int64_t r = blk * G + g;
        const bool valid = r < R;
        const T* row = z + (valid ? r : 0) * int64_t(K);
        const float lse = row_lse<TPR>(row, K, lane, valid);
        if (valid && lane == 0) {
            const int64_t y = labels[r % B];
            const float loss = (y >= 0 && y < K) ? lse - ldz(row, y) : qnan();
            if (lse_out) lse_out[r] = lse;
            acc += static_cast<double>(loss);
        }
    }
    __shared__ double red[G];
    if (lane == 0) red[g] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int i = 0; i < G; ++i) t += red[i];
        partials[blockIdx.x] = t;
    }
}

__global__ void __launch_bounds__(kThreads) categorical_total_kernel(const double* __restrict__ partials, int64_t n, float* __restrict__ total)
{
    __shared__ double red[kThreads];
    double t = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += kThreads) t += partials[i];
    red[threadIdx.x] = t;
    __syncthreads();
    for (int o = kThreads / 2; o > 0; o >>= 1) {
        if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) total[0] = static_cast<float>(red[0]);
}

template <int TPR, typename T>
__global__ void __launch_bounds__(kThreads)
categorical_nll_bwd_kernel(const T* __restrict__ z, const int64_t* __restrict__ labels, const float* __restrict__ lse,
                           const float* __restrict__ coef, T* __restrict__ dz, int64_t R, int64_t B, int K)
{
    constexpr int G = kThreads / TPR;
    const int g = threadIdx.x / TPR, lane = threadIdx.x % TPR;
    const float c = coef ? __ldg(coef) : 1.f;
    const int64_t blocks = (R + G - 1) / G;
    for (int64_t blk = blockIdx.x; blk < blocks; blk += gridDim.x) {
        const int64_t r = blk * G + g;
        if (r >= R) continue;
        const int64_t y = labels[r % B];
        const bool ok = y >= 0 && y < K;
        const float l = lse[r];
        const int64_t base = r * int64_t(K);
#pragma unroll 4
        for (int k = lane; k < K; k += TPR) {
            const float v = ok ? c * (expf(ldz(z, base + k) - l) - (k == y ? 1.f : 0.f)) : qnan();
            stz(dz, base + k, v);
        }
    }
}

template <int TPR, typename T>
__global__ void __launch_bounds__(kThreads)
categorical_predictive_kernel(const T* __restrict__ z, int64_t sample_stride, const int64_t* __restrict__ labels,
                              float* __restrict__ prob_sum, float* __restrict__ loglik_sum, int64_t S, int64_t B, int K,
                              int accumulate)
{
    constexpr int G = kThreads / TPR;
    const int g = threadIdx.x / TPR, lane = threadIdx.x % TPR;
    const int64_t blocks = (B + G - 1) / G;
    for (int64_t blk = blockIdx.x; blk < blocks; blk += gridDim.x) {   // CTA-uniform trip counts (row_lse may synchronise)
        const int64_t b = blk * G + g;
        const bool valid = b < B;
        const int64_t off = (valid ? b : 0) * int64_t(K);
        float* prow = prob_sum + off;
        int64_t y = 0;
        bool ok = false;
        if (valid && labels) {
            y = labels[b];
            ok = y >= 0 && y < K;
        }
        float ll = (accumulate && valid && loglik_sum) ? loglik_sum[b] : 0.f;
        for (int64_t s = 0; s < S; ++s) {
            const T* row = z + s * sample_stride + off;
            const float l = row_lse<TPR>(row, K, lane, valid);
            if (!valid) continue;
            const bool fresh = s == 0 && !accumulate;
            for (int k = lane; k < K; k += TPR) prow[k] = (fresh ? 0.f : prow[k]) + expf(ldz(row, k) - l);
            if (labels && lane == 0) ll += ok ? ldz(row, y) - l : qnan();
        }
        if (!valid) continue;
        if (S == 0 && !accumulate)
            for (int k = lane; k < K; k += TPR) prow[k] = 0.f;
        if (loglik_sum && lane == 0) loglik_sum[b] = ll;
    }
}

struct Plan {
    int tpr;
    int64_t ctas;
};

Plan plan(int64_t rows, int64_t K)
{
    int tpr = 2;
    while (tpr < K && tpr < 32) tpr <<= 1;
    if (K > 2048) tpr = kThreads;
    const int64_t per_cta = kThreads / tpr;
    int64_t ctas = (rows + per_cta - 1) / per_cta;
    ctas = ctas < 1 ? 1 : (ctas > kMaxCtas ? kMaxCtas : ctas);
    return {tpr, ctas};
}

// f(std::integral_constant<int, TPR>) for the plan's TPR
template <class F>
void with_tpr(int tpr, F&& f)
{
    switch (tpr) {
        case 2: f(std::integral_constant<int, 2>{}); break;
        case 4: f(std::integral_constant<int, 4>{}); break;
        case 8: f(std::integral_constant<int, 8>{}); break;
        case 16: f(std::integral_constant<int, 16>{}); break;
        case 32: f(std::integral_constant<int, 32>{}); break;
        default: f(std::integral_constant<int, kThreads>{}); break;
    }
}

template <typename T>
int nll_t(const void* z, const int64_t* labels, float* lse, float* total, void* ws, int64_t S, int64_t B, int64_t K, cudaStream_t st)
{
    const int64_t R = S * B;
    const Plan p = plan(R, K);
    double* partials = static_cast<double*>(ws);
    with_tpr(p.tpr, [&](auto tpr) {
        categorical_nll_kernel<decltype(tpr)::value, T><<<static_cast<unsigned>(p.ctas), kThreads, 0, st>>>(
            static_cast<const T*>(z), labels, lse, partials, R, B, static_cast<int>(K));
    });
    if (int rc = check_launch("categorical_nll_kernel")) return rc;
    categorical_total_kernel<<<1, kThreads, 0, st>>>(partials, p.ctas, total);
    return check_launch("categorical_total_kernel");
}

template <typename T>
int nll_bwd_t(const void* z, const int64_t* labels, const float* lse, const float* c, void* dz, int64_t S, int64_t B, int64_t K,
              cudaStream_t st)
{
    const int64_t R = S * B;
    if (R == 0) return WHVI_OK;
    const Plan p = plan(R, K);
    with_tpr(p.tpr, [&](auto tpr) {
        categorical_nll_bwd_kernel<decltype(tpr)::value, T><<<static_cast<unsigned>(p.ctas), kThreads, 0, st>>>(
            static_cast<const T*>(z), labels, lse, c, static_cast<T*>(dz), R, B, static_cast<int>(K));
    });
    return check_launch("categorical_nll_bwd_kernel");
}

template <typename T>
int predictive_t(const void* z, int64_t sample_stride, const int64_t* labels, float* prob_sum, float* loglik_sum, int64_t S, int64_t B,
                 int64_t K, int accumulate, cudaStream_t st)
{
    if (B == 0) return WHVI_OK;
    const Plan p = plan(B, K);
    with_tpr(p.tpr, [&](auto tpr) {
        categorical_predictive_kernel<decltype(tpr)::value, T><<<static_cast<unsigned>(p.ctas), kThreads, 0, st>>>(
            static_cast<const T*>(z), sample_stride, labels, prob_sum, loglik_sum, S, B, static_cast<int>(K), accumulate);
    });
    return check_launch("categorical_predictive_kernel");
}

}  // namespace

size_t categorical_workspace_bytes(int64_t R, int64_t K) { return sizeof(double) * static_cast<size_t>(plan(R, K).ctas); }

int launch_categorical_nll(const void* z, const int64_t* labels, float* lse, float* total, void* ws, int64_t S, int64_t B, int64_t K,
                           int bf16, cudaStream_t st)
{
    return bf16 ? nll_t<__nv_bfloat16>(z, labels, lse, total, ws, S, B, K, st) : nll_t<float>(z, labels, lse, total, ws, S, B, K, st);
}

int launch_categorical_nll_bwd(const void* z, const int64_t* labels, const float* lse, const float* c, void* dz, int64_t S, int64_t B,
                               int64_t K, int bf16, cudaStream_t st)
{
    return bf16 ? nll_bwd_t<__nv_bfloat16>(z, labels, lse, c, dz, S, B, K, st) : nll_bwd_t<float>(z, labels, lse, c, dz, S, B, K, st);
}

int launch_categorical_predictive(const void* z, int64_t sample_stride, const int64_t* labels, float* prob_sum, float* loglik_sum,
                                  int64_t S, int64_t B, int64_t K, int accumulate, int bf16, cudaStream_t st)
{
    return bf16 ? predictive_t<__nv_bfloat16>(z, sample_stride, labels, prob_sum, loglik_sum, S, B, K, accumulate, st)
                : predictive_t<float>(z, sample_stride, labels, prob_sum, loglik_sum, S, B, K, accumulate, st);
}

}  // namespace whvi
