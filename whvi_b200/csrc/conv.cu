// Patch gather and scatter of the convolutional WHVI layer (WHVIConv2d, not in the reference):
//   im2col   patches[s, (b, oh, ow), (i * kw + j) * C + c] = x[s, b, oh * sh - ph + i * dh, ow * sw - pw + j * dw, c]
//            (0 outside the image and in the columns n_in ... ld - 1, n_in = C * kh * kw): every element is written
//   col2im   dx[s, b, h, w, c] = sum over the taps (i, j) that read (h, w), i ascending then j ascending, of the matching
//            element of dpatches; with sum_samples the per-sample sums are added over s ascending into one (B, H, W, C) dx
// Activations are channels-last: x and dx (S|1, B, H, W, C), patches (S|1, B * Ho * Wo, ld), so the patch rows are the rows
// of the layer kernels and channels are the fastest axis of both sides.
//
// Work split (both kernels): a group of TPR threads (a power of two up to the CTA) walks the VEC-wide column vectors of a
// row (im2col: columns of a patch row; col2im: channels of a pixel), the CTA holds 256 / TPR such groups, and the groups
// stride over the rows with a position (s, b, oh, ow) advanced by carries instead of divided out per row.  A column vector
// is 16 bytes (4 fp32 or 8 bf16 channels) when the channel runs and both base pointers allow it, one element otherwise.
// im2col is a copy of words (the bf16 instance moves the same bits as the fp32 one); col2im adds in fp32 and rounds a bf16
// dx once.  No atomics: every output element is owned by one thread, so both are bit-reproducible.
#include <cuda_bf16.h>

#include <type_traits>

#include "common.cuh"

namespace whvi {
namespace {

constexpr int kThreads = 256;
constexpr int64_t kMaxCtas = 148 * 8;   // one resident wave of 256-thread CTAs
constexpr int kRowsInFlight = 4;        // independent loads per thread per round (bandwidth: bytes in flight per SM)

// r = ((s * B + b) * P + p) * Q + q: a row (im2col: p, q = oh, ow) or a pixel (col2im: p, q = h, w)
struct Pos {
    int64_t s, b;
    int p, q;
};

__device__ __forceinline__ Pos decode(int64_t r, int64_t B, int P, int Q)
{
    Pos o;
    int64_t t = r / Q;
    o.q = static_cast<int>(r - t * Q);
    const int64_t u = t / P;
    o.p = static_cast<int>(t - u * P);
    o.s = u / B;
    o.b = u - o.s * B;
    return o;
}

// a += d for positions with every component below its modulus (so each carry is 0 or 1)
__device__ __forceinline__ void advance(Pos& a, const Pos& d, int64_t B, int P, int Q)
{
    a.q += d.q;
    int c = a.q >= Q;
    a.q -= c * Q;
    a.p += d.p + c;
    c = a.p >= P;
    a.p -= c * P;
    a.b += d.b + c;
    const int64_t cb = a.b >= B;
    a.b -= cb * B;
    a.s += d.s + cb;
}

int tpr_for(int64_t vecs)
{
    int t = 1;
    while (t < vecs && t < kThreads) t <<= 1;
    return t;
}

// E: the element's bits (uint32_t for fp32, uint16_t for bf16); V: one move of VEC elements
template <typename E, int VEC>
__global__ void __launch_bounds__(kThreads)
im2col_kernel(const E* __restrict__ x, int64_t xs, E* __restrict__ out, ConvGeom g, int64_t ld, int64_t n_in, int tpr)
{
    using V = typename std::conditional<VEC == 1, E, uint4>::type;
    const int rpc = kThreads / tpr;
    const int sub = threadIdx.x % tpr;
    const int64_t rows = g.S * g.B * g.Ho * g.Wo;
    const int64_t step = int64_t(gridDim.x) * rpc;
    const int64_t r0 = int64_t(blockIdx.x) * rpc + threadIdx.x / tpr;
    if (r0 >= rows) return;
    const Pos d = decode(step, g.B, g.Ho, g.Wo);
    const int64_t img = int64_t(g.H) * g.W * g.C;
    for (int64_t col = int64_t(sub) * VEC; col < ld; col += int64_t(tpr) * VEC) {
        const bool live = col < n_in;   // n_in % VEC == 0 on the vector path: a move is all taps or all padding
        const int tap = static_cast<int>(col / g.C), c = static_cast<int>(col - int64_t(tap) * g.C);
        const int i = tap / g.kw, j = tap - i * g.kw;
        const int di = i * g.dh - g.ph, dj = j * g.dw - g.pw;
        Pos p = decode(r0, g.B, g.Ho, g.Wo);
        for (int64_t r = r0; r < rows;) {
            V v[kRowsInFlight];
            int64_t at[kRowsInFlight];
#pragma unroll
            for (int k = 0; k < kRowsInFlight; ++k) {
                v[k] = V{};
                at[k] = r;
                const int ih = p.p * g.sh + di, iw = p.q * g.sw + dj;
                if (live && r < rows && ih >= 0 && ih < g.H && iw >= 0 && iw < g.W)
                    v[k] = __ldg(reinterpret_cast<const V*>(x + p.s * xs + p.b * img + (int64_t(ih) * g.W + iw) * g.C + c));
                r += step;
                advance(p, d, g.B, g.Ho, g.Wo);
            }
#pragma unroll
            for (int k = 0; k < kRowsInFlight; ++k)
                if (at[k] < rows) *reinterpret_cast<V*>(out + at[k] * ld + col) = v[k];
        }
    }
}

template <typename T>
__device__ __forceinline__ float widen(T v)
{
    if constexpr (std::is_same<T, float>::value) return v;
    else return __bfloat162float(v);
}

// acc[0 .. VEC) += p[0 .. VEC)
template <typename T, int VEC>
__device__ __forceinline__ void add_from(float* acc, const T* p)
{
    if constexpr (VEC == 1) {
        acc[0] += widen(p[0]);
    } else if constexpr (std::is_same<T, float>::value) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(p));
        acc[0] += v.x;
        acc[1] += v.y;
        acc[2] += v.z;
        acc[3] += v.w;
    } else {
        const uint4 v = __ldg(reinterpret_cast<const uint4*>(p));   // bf16 pairs: element 2k in the low half of word k
        acc[0] += __uint_as_float(v.x << 16);
        acc[1] += __uint_as_float(v.x & 0xffff0000u);
        acc[2] += __uint_as_float(v.y << 16);
        acc[3] += __uint_as_float(v.y & 0xffff0000u);
        acc[4] += __uint_as_float(v.z << 16);
        acc[5] += __uint_as_float(v.z & 0xffff0000u);
        acc[6] += __uint_as_float(v.w << 16);
        acc[7] += __uint_as_float(v.w & 0xffff0000u);
    }
}

__device__ __forceinline__ uint32_t bf16_pair(float lo, float hi)
{
    return uint32_t(__bfloat16_as_ushort(__float2bfloat16_rn(lo))) | (uint32_t(__bfloat16_as_ushort(__float2bfloat16_rn(hi))) << 16);
}

template <typename T, int VEC>
__device__ __forceinline__ void store(T* p, const float* v)
{
    if constexpr (VEC == 1) {
        if constexpr (std::is_same<T, float>::value) p[0] = v[0];
        else p[0] = __float2bfloat16_rn(v[0]);
    } else if constexpr (std::is_same<T, float>::value) {
        *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
    } else {
        *reinterpret_cast<uint4*>(p) = make_uint4(bf16_pair(v[0], v[1]), bf16_pair(v[2], v[3]), bf16_pair(v[4], v[5]), bf16_pair(v[6], v[7]));
    }
}

// one thread per (pixel, channel vector) of dx; the taps that read pixel (h, w) are those with h + ph - i * dh = oh * sh,
// 0 <= oh < Ho (likewise w), visited i ascending, j ascending
template <typename T, int VEC>
__global__ void __launch_bounds__(kThreads, 2)
col2im_kernel(const T* __restrict__ dp, int64_t ld, T* __restrict__ dx, ConvGeom g, int sum_samples, int tpr)
{
    const int rpc = kThreads / tpr;
    const int sub = threadIdx.x % tpr;
    const int64_t S_out = sum_samples ? 1 : g.S;
    const int64_t pixels = S_out * g.B * g.H * g.W;
    const int64_t step = int64_t(gridDim.x) * rpc;
    const int64_t r0 = int64_t(blockIdx.x) * rpc + threadIdx.x / tpr;
    if (r0 >= pixels) return;
    const Pos d = decode(step, g.B, g.H, g.W);
    for (int c = sub * VEC; c < g.C; c += tpr * VEC) {
        Pos p = decode(r0, g.B, g.H, g.W);
        for (int64_t r = r0; r < pixels; r += step, advance(p, d, g.B, g.H, g.W)) {
            float tot[VEC];
#pragma unroll
            for (int k = 0; k < VEC; ++k) tot[k] = 0.f;
            const int64_t s_end = sum_samples ? g.S : p.s + 1;
            for (int64_t s = sum_samples ? 0 : p.s; s < s_end; ++s) {
                float acc[VEC];
#pragma unroll
                for (int k = 0; k < VEC; ++k) acc[k] = 0.f;
                const T* base = dp + (s * g.B + p.b) * g.Ho * g.Wo * ld + c;
                for (int i = 0; i < g.kh; ++i) {
                    const int th = p.p + g.ph - i * g.dh;
                    if (th < 0) break;   // th only falls with i
                    const int oh = th / g.sh;
                    if (oh * g.sh != th || oh >= g.Ho) continue;
                    for (int j = 0; j < g.kw; ++j) {
                        const int tw = p.q + g.pw - j * g.dw;
                        if (tw < 0) break;
                        const int ow = tw / g.sw;
                        if (ow * g.sw != tw || ow >= g.Wo) continue;
                        add_from<T, VEC>(acc, base + (int64_t(oh) * g.Wo + ow) * ld + int64_t(i * g.kw + j) * g.C);
                    }
                }
                if (sum_samples) {
#pragma unroll
                    for (int k = 0; k < VEC; ++k) tot[k] += acc[k];
                } else {
#pragma unroll
                    for (int k = 0; k < VEC; ++k) tot[k] = acc[k];
                }
            }
            store<T, VEC>(dx + ((p.s * g.B + p.b) * g.H * g.W + int64_t(p.p) * g.W + p.q) * g.C + c, tot);
        }
    }
}

template <typename E, int VEC>
int im2col_t(const void* x, int64_t xs, void* out, const ConvGeom& g, int64_t ld, cudaStream_t st)
{
    const int64_t rows = g.S * g.B * g.Ho * g.Wo;
    const int tpr = tpr_for(ld / VEC);
    const int64_t rpc = kThreads / tpr;
    int64_t ctas = (rows + rpc - 1) / rpc;
    ctas = ctas > kMaxCtas ? kMaxCtas : ctas;
    im2col_kernel<E, VEC><<<static_cast<unsigned>(ctas), kThreads, 0, st>>>(static_cast<const E*>(x), xs, static_cast<E*>(out), g, ld,
                                                                         int64_t(g.C) * g.kh * g.kw, tpr);
    return check_launch("im2col_kernel");
}

template <typename T, int VEC>
int col2im_t(const void* dp, int64_t ld, void* dx, const ConvGeom& g, int sum_samples, cudaStream_t st)
{
    const int64_t pixels = (sum_samples ? 1 : g.S) * g.B * g.H * g.W;
    const int tpr = tpr_for(g.C / VEC);
    const int64_t rpc = kThreads / tpr;
    int64_t ctas = (pixels + rpc - 1) / rpc;
    ctas = ctas > kMaxCtas ? kMaxCtas : ctas;
    col2im_kernel<T, VEC><<<static_cast<unsigned>(ctas), kThreads, 0, st>>>(static_cast<const T*>(dp), ld, static_cast<T*>(dx), g,
                                                                         sum_samples, tpr);
    return check_launch("col2im_kernel");
}

}  // namespace

int launch_im2col(const void* x, int64_t xs, void* out, const ConvGeom& g, int64_t ld, int bf16, cudaStream_t st)
{
    if (g.S * g.B == 0) return WHVI_OK;
    const int vec = bf16 ? 8 : 4;
    const bool wide = g.C % vec == 0 && ld % vec == 0 && xs % vec == 0 && aligned16(x) && aligned16(out);
    if (bf16) return wide ? im2col_t<uint16_t, 8>(x, xs, out, g, ld, st) : im2col_t<uint16_t, 1>(x, xs, out, g, ld, st);
    return wide ? im2col_t<uint32_t, 4>(x, xs, out, g, ld, st) : im2col_t<uint32_t, 1>(x, xs, out, g, ld, st);
}

int launch_col2im(const void* dp, int64_t ld, void* dx, const ConvGeom& g, int sum_samples, int bf16, cudaStream_t st)
{
    if ((sum_samples ? 1 : g.S) * g.B == 0) return WHVI_OK;
    const int vec = bf16 ? 8 : 4;
    const bool wide = g.C % vec == 0 && ld % vec == 0 && aligned16(dp) && aligned16(dx);
    if (bf16)
        return wide ? col2im_t<__nv_bfloat16, 8>(dp, ld, dx, g, sum_samples, st) : col2im_t<__nv_bfloat16, 1>(dp, ld, dx, g, sum_samples, st);
    return wide ? col2im_t<float, 4>(dp, ld, dx, g, sum_samples, st) : col2im_t<float, 1>(dp, ld, dx, g, sum_samples, st);
}

}  // namespace whvi
