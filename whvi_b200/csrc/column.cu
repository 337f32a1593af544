// WHVIColumnMatrix (src/weights.py:211-251), PAPER semantics, as one call per direction.
//
// The reference samples the whole D x D matrix (four FWHTs of D x D matrices, src/weights.py:66-73), flattens it and keeps
// the first n entries (:239-245) -- row 0 of W = S1 H diag(g) H S2:
//     w[s, j] = s1[0] * s2[j] * (H g_s)[j],   j < n,    g_s = mu + softplus(rho) * eps_s
// so one FWHT of g per MC sample is all the transform work there is.  The layer is then a 1-wide product:
//     transposed (n_in = n, n_out = 1):  y[s, b]    = sum_j x[s, b, j] w[s, j] + bias          (src/weights.py:247-249)
//     plain      (n_in = 1, n_out = n):  y[s, b, j] = x[s, b] w[s, j] + bias[j]
// Everything here is HBM-bound elementwise / reduction work on the activations (4 B per element each way); the weights
// (S x D) are noise next to them.  All reductions have a fixed order (bit-reproducible).
//
// bf16 activations (A = __nv_bfloat16): x, dx and -- plain form only -- y and dy are bf16 in HBM; g, H g, the parameters,
// their gradients and every sum stay fp32.  Each value is widened on load and rounded once at the store, and the reduction
// orders are the fp32 kernels', so a bf16 call is the fp32 call on the widened inputs with its activation outputs rounded.
// The transposed form's output y (S, B, 1) and its gradient dy stay fp32: 1/n of the input's bytes, and rounding the
// network's predictions would put that error straight into the loss.
#include "common.cuh"
#include "engine.cuh"

namespace whvi {

__device__ __forceinline__ float widen(float v) { return v; }
__device__ __forceinline__ float widen(__nv_bfloat16 v) { return __bfloat162float(v); }
template <class T>
__device__ __forceinline__ T narrow(float v);
template <>
__device__ __forceinline__ float narrow<float>(float v) { return v; }
template <>
__device__ __forceinline__ __nv_bfloat16 narrow<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// ---- forward ---------------------------------------------------------------------------------------------------------
// transposed: one warp per (s, b) row; w is formed on the fly from hg = H g (L2-resident)
template <class A>
__global__ void __launch_bounds__(256)
column_dot_kernel(const A* __restrict__ x, int64_t xs, const float* __restrict__ hg, const float* __restrict__ s1, const float* __restrict__ s2,
                  const float* __restrict__ bias, float* __restrict__ y, int64_t S, int64_t B, int D, int n)
{
    const int64_t row = int64_t(blockIdx.x) * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= S * B) return;
    const int64_t s = row / B, b = row - s * B;
    const A* xr = x + s * xs + b * n;
    const float* h = hg + s * D;
    float acc = 0.f;
    for (int j = lane; j < n; j += 32) acc = fmaf(widen(xr[j]), s2[j] * h[j], acc);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) y[row] = fmaf(acc, s1[0], bias ? bias[0] : 0.f);
}

// plain: y[s, b, j] = x[s, b] * w[s, j] + bias[j]
template <class A>
__global__ void __launch_bounds__(256)
column_outer_kernel(const A* __restrict__ x, int64_t xs, const float* __restrict__ hg, const float* __restrict__ s1,
                    const float* __restrict__ s2, const float* __restrict__ bias, A* __restrict__ y, int64_t S, int64_t B, int D, int n, int relu_out)
{
    const int64_t total = S * B * n;
    const float a = s1[0];
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += int64_t(gridDim.x) * blockDim.x) {
        const int j = static_cast<int>(i % n);
        const int64_t row = i / n, s = row / B, b = row - s * B;
        float v = fmaf(widen(x[s * xs + b]), a * s2[j] * hg[s * D + j], bias ? bias[j] : 0.f);
        if (relu_out) v = fmaxf(v, 0.f);
        y[i] = narrow<A>(v);
    }
}

// ---- backward ----------------------------------------------------------------------------------------------------------
// transposed: dx[s, b, j] = dy[s, b] w[s, j] (x (x > 0) when the input is the output of a fused ReLU)
template <class A>
__global__ void __launch_bounds__(256)
column_dot_dx_kernel(const float* __restrict__ dy, const A* __restrict__ x, int64_t xs, const float* __restrict__ hg, const float* __restrict__ s1,
                     const float* __restrict__ s2, A* __restrict__ dx, int64_t S, int64_t B, int D, int n, int relu_in)
{
    const int64_t total = S * B * n;
    const float a = s1[0];
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += int64_t(gridDim.x) * blockDim.x) {
        const int j = static_cast<int>(i % n);
        const int64_t row = i / n, s = row / B, b = row - s * B;
        float v = dy[row] * (a * s2[j] * hg[s * D + j]);
        if (relu_in && !(widen(x[s * xs + b * n + j]) > 0.f)) v = 0.f;
        dx[i] = narrow<A>(v);
    }
}

// dwp[s, j] = sum_b u[s, b] * v[s, b, j] over the batch: transposed u = dy (S, B), v = x (S, B, n); plain u = x (S, B), v = dy (S, B, n).
// 32 columns x 8 batch slices per CTA, slices combined in a fixed order.  grid (ceil(n / 32), min(S, 65535)); a CTA takes samples
// blockIdx.y, + gridDim.y, ...  U, V: the activation types of u, v.
template <class U, class V>
__global__ void __launch_bounds__(256)
column_dw_kernel(const U* __restrict__ u, int64_t us, const V* __restrict__ v, int64_t vs, float* __restrict__ dwp, int64_t S, int64_t B, int n)
{
    __shared__ float red[8][32];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int j = blockIdx.x * 32 + tx;
    for (int64_t s = blockIdx.y; s < S; s += gridDim.y) {
        const U* up = u + s * us;
        const V* vp = v + s * vs;
        float acc = 0.f;
        if (j < n)
            for (int64_t b = ty; b < B; b += 8) acc = fmaf(widen(up[b]), widen(vp[b * n + j]), acc);
        red[ty][tx] = acc;
        __syncthreads();
        if (ty == 0 && j < n) {
#pragma unroll
            for (int q = 1; q < 8; ++q) acc += red[q][tx];
            dwp[s * n + j] = acc;
        }
        __syncthreads();   // red is refilled for the next sample
    }
}

// plain: dx[s, b] = sum_j dy[s, b, j] w[s, j]; one warp per row
template <class A>
__global__ void __launch_bounds__(256)
column_outer_dx_kernel(const A* __restrict__ dy, const float* __restrict__ hg, const float* __restrict__ s1, const float* __restrict__ s2,
                       A* __restrict__ dx, int64_t S, int64_t B, int D, int n)
{
    const int64_t row = int64_t(blockIdx.x) * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= S * B) return;
    const int64_t s = row / B;
    const A* d = dy + row * n;
    const float* h = hg + s * D;
    float acc = 0.f;
    for (int j = lane; j < n; j += 32) acc = fmaf(widen(d[j]), s2[j] * h[j], acc);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) dx[row] = narrow<A>(acc * s1[0]);
}

// dbias[c] = sum over rows of dy[row, c] (cols = 1 transposed, n plain): one CTA per 32 columns, fixed order
template <class A>
__global__ void __launch_bounds__(256)
column_dbias_kernel(const A* __restrict__ dy, float* __restrict__ dbias, int64_t rows, int cols)
{
    __shared__ float red[8][32];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    float acc = 0.f;
    if (cols == 1) {   // a plain sum: all 256 threads stride the rows
        for (int64_t r = threadIdx.x; r < rows; r += 256) acc += widen(dy[r]);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (tx == 0) red[ty][0] = acc;
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int q = 1; q < 8; ++q) acc += red[q][0];
            dbias[0] = acc;
        }
        return;
    }
    const int c = blockIdx.x * 32 + tx;
    if (c < cols)
        for (int64_t r = ty; r < rows; r += 8) acc += widen(dy[r * cols + c]);
    red[ty][tx] = acc;
    __syncthreads();
    if (ty == 0 && c < cols) {
#pragma unroll
        for (int q = 1; q < 8; ++q) acc += red[q][tx];
        dbias[c] = acc;
    }
}

// From dwp[s, j] = dL/dw[s, j] to the parameter side:  dhg[s, j] = dwp * s1[0] * s2[j] (zero for j >= n),
// q[j] = sum_s dwp[s, j] * hg[s, j]  ->  ds2[j] = s1[0] * q[j] (zero for j >= n), and ds1[0] = sum_j s2[j] q[j] by a last block
// (fixed order: a single thread block folds the per-block partial sums written to `part`).
__global__ void __launch_bounds__(256)
column_param_kernel(const float* __restrict__ dwp, const float* __restrict__ hg, const float* __restrict__ s1, const float* __restrict__ s2,
                    float* __restrict__ dhg, float* __restrict__ ds2, float* __restrict__ part, int64_t S, int D, int n)
{
    __shared__ float red[8];
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    const float a = s1[0];
    float contrib = 0.f;
    if (j < D) {
        float q = 0.f;
        const float sj = j < n ? s2[j] : 0.f;
        for (int64_t s = 0; s < S; ++s) {
            const float d = j < n ? dwp[s * n + j] : 0.f;
            q = fmaf(d, hg[s * D + j], q);
            dhg[s * D + j] = d * a * sj;
        }
        ds2[j] = a * q;
        contrib = sj * q;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) contrib += __shfl_xor_sync(0xffffffffu, contrib, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = contrib;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.f;
        for (int w = 0; w < 8; ++w) t += red[w];
        part[blockIdx.x] = t;
    }
}
__global__ void column_ds1_kernel(const float* __restrict__ part, int nparts, float* __restrict__ ds1, int D)
{
    for (int i = threadIdx.x; i < D; i += blockDim.x) ds1[i] = 0.f;   // only s1[0] enters row 0 of W
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.f;
        for (int i = 0; i < nparts; ++i) t += part[i];
        ds1[0] = t;
    }
}

static unsigned ew_grid(int64_t total)
{
    int64_t b = (total + 255) / 256;
    if (b > 148 * 16) b = 148 * 16;
    return static_cast<unsigned>(b < 1 ? 1 : b);
}

template <class A>
static int column_fwd_product(const float* x, int64_t xs, const float* hg, const float* s1, const float* s2, const float* bias, float* y,
                              int64_t S, int64_t B, int64_t D, int64_t n, int transposed, int relu_out, cudaStream_t st)
{
    const A* xa = reinterpret_cast<const A*>(x);
    if (transposed) {
        const int64_t blocks = (S * B + 7) / 8;
        if (blocks > 0x7fffffffLL) return fail(WHVI_E_SHAPE, "column_fwd: too many rows");
        column_dot_kernel<A><<<static_cast<unsigned>(blocks), 256, 0, st>>>(xa, xs, hg, s1, s2, bias, y, S, B, static_cast<int>(D), static_cast<int>(n));
        return check_launch("column_dot_kernel");
    }
    column_outer_kernel<A><<<ew_grid(S * B * n), 256, 0, st>>>(xa, xs, hg, s1, s2, bias, reinterpret_cast<A*>(y), S, B, static_cast<int>(D),
                                                               static_cast<int>(n), relu_out);
    return check_launch("column_outer_kernel");
}

// the layer from g (S, D), however g was drawn: hg = H g, then the 1-wide product.  bf16: x (and the plain form's y) are bf16
// behind the float pointers; the transposed form's y stays fp32.
int launch_column_fwd_g(const float* x, int64_t xs, const float* g, const float* s1, const float* s2, const float* bias, float* hg, float* y,
                        int64_t S, int64_t B, int64_t D, int64_t n, int transposed, int relu_out, cudaStream_t st, int bf16)
{
    if (int rc = launch_fwht(g, hg, S, D, st)) return rc;
    return bf16 ? column_fwd_product<__nv_bfloat16>(x, xs, hg, s1, s2, bias, y, S, B, D, n, transposed, relu_out, st)
                : column_fwd_product<float>(x, xs, hg, s1, s2, bias, y, S, B, D, n, transposed, relu_out, st);
}

int launch_column_fwd(const float* x, int64_t xs, const float* mu, const float* rho, const float* s1, const float* s2, const float* eps,
                      const float* bias, float* g, float* hg, float* y, int64_t S, int64_t B, int64_t D, int64_t n, int transposed, int relu_out,
                      cudaStream_t st, int bf16)
{
    if (int rc = launch_reparam_diag(mu, rho, eps, g, S, D, st)) return rc;
    return launch_column_fwd_g(x, xs, g, s1, s2, bias, hg, y, S, B, D, n, transposed, relu_out, st, bf16);
}

static int64_t up4(int64_t v) { return (v + 3) / 4 * 4; }   // every segment starts 16-byte aligned (the FWHT reads float4s)

size_t column_bwd_workspace_bytes(int64_t S, int64_t D, int64_t n)
{
    // dhg (S, D) | dg (S, D) | dwp (S, n) | partial sums (ceil(D / 256))
    return sizeof(float) * size_t(2 * up4(S * D) + up4(S * n) + up4((D + 255) / 256));
}

// the activation side of the backward: dx and dwp (S, n) = dL/dw, and dbias
template <class A>
static int column_bwd_products(const float* x, int64_t xs, const float* dy, const float* hg, const float* s1, const float* s2, float* dx,
                               float* dbias, float* dwp, int64_t S, int64_t B, int64_t D, int64_t n, int transposed, int relu_in, cudaStream_t st)
{
    const A* xa = reinterpret_cast<const A*>(x);
    A* dxa = reinterpret_cast<A*>(dx);
    const int Di = static_cast<int>(D), ni = static_cast<int>(n);
    const dim3 dwgrid(static_cast<unsigned>((n + 31) / 32), static_cast<unsigned>(S < 65535 ? S : 65535));   // grid.y <= 65535
    if (transposed) {   // dy (S, B) is fp32
        if (dx) {
            column_dot_dx_kernel<A><<<ew_grid(S * B * n), 256, 0, st>>>(dy, xa, xs, hg, s1, s2, dxa, S, B, Di, ni, relu_in);
            if (int rc = check_launch("column_dot_dx_kernel")) return rc;
        }
        column_dw_kernel<float, A><<<dwgrid, 256, 0, st>>>(dy, B, xa, xs, dwp, S, B, ni);   // u = dy (S, B), v = x (stride xs: 0 when shared)
    } else {
        const A* dya = reinterpret_cast<const A*>(dy);
        if (dx) {
            const int64_t blocks = (S * B + 7) / 8;
            column_outer_dx_kernel<A><<<static_cast<unsigned>(blocks), 256, 0, st>>>(dya, hg, s1, s2, dxa, S, B, Di, ni);
            if (int rc = check_launch("column_outer_dx_kernel")) return rc;
        }
        column_dw_kernel<A, A><<<dwgrid, 256, 0, st>>>(xa, xs, dya, B * n, dwp, S, B, ni);  // u = x (S, B) (stride xs), v = dy (S, B, n)
    }
    if (int rc = check_launch("column_dw_kernel")) return rc;
    if (dbias) {
        const int cols = transposed ? 1 : ni;
        if (transposed)
            column_dbias_kernel<float><<<1, 256, 0, st>>>(dy, dbias, S * B, cols);
        else
            column_dbias_kernel<A><<<static_cast<unsigned>((cols + 31) / 32), 256, 0, st>>>(reinterpret_cast<const A*>(dy), dbias, S * B, cols);
        if (int rc = check_launch("column_dbias_kernel")) return rc;
    }
    return WHVI_OK;
}

// the layer's backward down to dg (S, D); ws as column_bwd_workspace_bytes (its dg segment stays unused when dg is the caller's).
// bf16: x, dx (and the plain form's dy) are bf16 behind the float pointers; the transposed form's dy stays fp32.
int launch_column_bwd_g(const float* x, int64_t xs, const float* dy, const float* hg, const float* s1, const float* s2, float* dx, float* dg,
                        float* ds1, float* ds2, float* dbias, float* ws, int64_t S, int64_t B, int64_t D, int64_t n, int transposed, int relu_in,
                        cudaStream_t st, int bf16)
{
    float* dhg = ws;
    float* dwp = dhg + 2 * up4(S * D);
    float* part = dwp + up4(S * n);
    const int Di = static_cast<int>(D), ni = static_cast<int>(n);
    if (int rc = bf16 ? column_bwd_products<__nv_bfloat16>(x, xs, dy, hg, s1, s2, dx, dbias, dwp, S, B, D, n, transposed, relu_in, st)
                      : column_bwd_products<float>(x, xs, dy, hg, s1, s2, dx, dbias, dwp, S, B, D, n, transposed, relu_in, st))
        return rc;
    const int nparts = static_cast<int>((D + 255) / 256);
    column_param_kernel<<<nparts, 256, 0, st>>>(dwp, hg, s1, s2, dhg, ds2, part, S, Di, ni);
    if (int rc = check_launch("column_param_kernel")) return rc;
    column_ds1_kernel<<<1, 256, 0, st>>>(part, nparts, ds1, Di);
    if (int rc = check_launch("column_ds1_kernel")) return rc;
    return launch_fwht(dhg, dg, S, D, st);   // dg = H dhg (H is symmetric)
}

int launch_column_bwd(const float* x, int64_t xs, const float* dy, const float* hg, const float* rho, const float* s1, const float* s2,
                      const float* eps, float* dx, float* dmu, float* drho, float* ds1, float* ds2, float* dbias, float* ws, int64_t S,
                      int64_t B, int64_t D, int64_t n, int transposed, int relu_in, cudaStream_t st, int bf16)
{
    float* dg = ws + up4(S * D);
    if (int rc = launch_column_bwd_g(x, xs, dy, hg, s1, s2, dx, dg, ds1, ds2, dbias, ws, S, B, D, n, transposed, relu_in, st, bf16)) return rc;
    return launch_reparam_diag_bwd(rho, eps, dg, dmu, drho, S, D, 0, st);
}

}  // namespace whvi
