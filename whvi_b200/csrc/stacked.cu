// WHVIStackedMatrix (src/weights.py:111-208) as ONE call per direction.
//
// The reference pads the input to D = next_pow2(n_in) columns (:197-198), runs its G = ceil(n_out / D) square blocks one
// after the other on the same padded input (:179-180), concatenates their outputs, adds the bias and drops the columns
// past n_out (:204-207).  Here the blocks are a second sample axis of the fused layer kernels ("virtual samples"
// s' = block * S + sample, each with its own g; s1 / s2 / bias are picked per block inside the kernels), so the whole
// stack is one reparameterisation launch, one layer launch and one interleave launch, whatever G is:
//
//   forward   [pad x]  ->  g = mu_k + softplus(rho_k) eps  ->  layer_fwd over G*S virtual samples  ->  y[s, b, k D + j]
//   backward  dy[s, b, k D + j] -> (G, S, B, D)  ->  layer_bwd (3 launches)  ->  reparam_bwd  ->  [dx = sum_k dx_k, unpadded]
//
// The bias (1, G*D) and the ReLU that follows the layer ride in the layer kernel (bias vector k D .. k D + D - 1 for
// block k).  Parameter vectors of block k are read at base + k * param_stride, so the blocks' separate nn.Parameters can
// be used where they lie as long as they are evenly spaced (they are once packed by FlatParams or by the module itself).
#include "common.cuh"
#include "engine.cuh"
#include <type_traits>

namespace whvi {

// T: the activation type, float or __nv_bfloat16.  Four consecutive elements move as one unit (16 bytes of fp32, 8 of bf16);
// split and concat are exact copies, so bf16 elements are moved as their bit patterns.
template <class T>
struct Lanes;
template <>
struct Lanes<float> {
    using V = float4;
    static __device__ __forceinline__ float4 zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }
    static __device__ __forceinline__ float get(const float4& v, int k) { return k == 0 ? v.x : k == 1 ? v.y : k == 2 ? v.z : v.w; }
    static __device__ __forceinline__ void set(float4& v, int k, float e) { (k == 0 ? v.x : k == 1 ? v.y : k == 2 ? v.z : v.w) = e; }
    static __device__ __forceinline__ float4 round(const float4& a) { return a; }
};
template <>
struct Lanes<__nv_bfloat16> {
    using V = uint2;   // element 2q in the low half of word q, 2q + 1 in the high half
    static __device__ __forceinline__ uint2 zero() { return make_uint2(0u, 0u); }
    static __device__ __forceinline__ __nv_bfloat16 get(const uint2& v, int k)
    {
        const uint32_t w = k < 2 ? v.x : v.y;
        return __ushort_as_bfloat16(static_cast<unsigned short>(k & 1 ? w >> 16 : w & 0xFFFFu));
    }
    static __device__ __forceinline__ void set(uint2& v, int k, __nv_bfloat16 e)
    {
        uint32_t& w = k < 2 ? v.x : v.y;
        const uint32_t b = __bfloat16_as_ushort(e);
        w = k & 1 ? (w & 0xFFFFu) | (b << 16) : (w & 0xFFFF0000u) | b;
    }
    static __device__ __forceinline__ uint2 round(const float4& a)   // round to nearest even, once
    {
        uint2 r;
        asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r.x) : "f"(a.y), "f"(a.x));
        asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r.y) : "f"(a.w), "f"(a.z));
        return r;
    }
};

// blocks (G, R, D) -> out (R, n_out), out[r, k D + j] = blocks[k, r, j] for k D + j < n_out      (R = S * B rows)
template <class T>
__global__ void __launch_bounds__(256)
stack_concat_kernel(const typename Lanes<T>::V* __restrict__ blocks, T* __restrict__ out, int64_t R, int D4, int64_t G, int64_t n_out, int vec)
{
    using L = Lanes<T>;
    const int64_t total = G * R * D4;
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += int64_t(gridDim.x) * blockDim.x) {
        const int j4 = static_cast<int>(i % D4);
        const int64_t kr = i / D4, r = kr % R, k = kr / R;
        const int64_t col = k * (int64_t(D4) * 4) + 4 * j4;
        if (col >= n_out) continue;
        const typename L::V v = blocks[i];
        T* o = out + r * n_out + col;
        if (vec) {
            *reinterpret_cast<typename L::V*>(o) = v;
        } else {
            o[0] = L::get(v, 0);
            if (col + 1 < n_out) o[1] = L::get(v, 1);
            if (col + 2 < n_out) o[2] = L::get(v, 2);
            if (col + 3 < n_out) o[3] = L::get(v, 3);
        }
    }
}

// the inverse: in (R, n_out) -> blocks (G, R, D), zero where k D + j >= n_out.  With G = 1 this is the zero-padding of the
// input rows to D columns.
template <class T>
__global__ void __launch_bounds__(256)
stack_split_kernel(const T* __restrict__ in, typename Lanes<T>::V* __restrict__ blocks, int64_t R, int D4, int64_t G, int64_t n_out, int vec)
{
    using L = Lanes<T>;
    const int64_t total = G * R * D4;
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += int64_t(gridDim.x) * blockDim.x) {
        const int j4 = static_cast<int>(i % D4);
        const int64_t kr = i / D4, r = kr % R, k = kr / R;
        const int64_t col = k * (int64_t(D4) * 4) + 4 * j4;
        typename L::V v = L::zero();
        if (col < n_out) {
            const T* p = in + r * n_out + col;
            if (vec) {
                v = *reinterpret_cast<const typename L::V*>(p);
            } else {
                L::set(v, 0, p[0]);
                if (col + 1 < n_out) L::set(v, 1, p[1]);
                if (col + 2 < n_out) L::set(v, 2, p[2]);
                if (col + 3 < n_out) L::set(v, 3, p[3]);
            }
        }
        blocks[i] = v;
    }
}

// dx[r, j] = sum_k dxb[k, r, j] for j < n_in (blocks ascending: fixed order); rows of dx are n_in wide.  dxb is fp32 for either T:
// the sum is taken in fp32 and rounded to T once, at the store.
template <class T>
__global__ void __launch_bounds__(256)
stack_sum_kernel(const float4* __restrict__ dxb, T* __restrict__ dx, int64_t R, int D4, int64_t G, int64_t n_in, int vec)
{
    using L = Lanes<T>;
    const int64_t total = R * D4;
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += int64_t(gridDim.x) * blockDim.x) {
        const int j4 = static_cast<int>(i % D4);
        const int64_t r = i / D4, col = 4 * int64_t(j4);
        if (col >= n_in) continue;
        float4 a = dxb[i];
        for (int64_t k = 1; k < G; ++k) {
            const float4 q = dxb[k * total + i];
            a.x += q.x, a.y += q.y, a.z += q.z, a.w += q.w;
        }
        const typename L::V v = L::round(a);
        T* o = dx + r * n_in + col;
        if (vec) {
            *reinterpret_cast<typename L::V*>(o) = v;
        } else {
            o[0] = L::get(v, 0);
            if (col + 1 < n_in) o[1] = L::get(v, 1);
            if (col + 2 < n_in) o[2] = L::get(v, 2);
            if (col + 3 < n_in) o[3] = L::get(v, 3);
        }
    }
}

static unsigned grid_for(int64_t total)
{
    int64_t b = (total + 255) / 256;
    if (b > 148 * 16) b = 148 * 16;
    return static_cast<unsigned>(b < 1 ? 1 : b);
}

// the vector path needs whole 4-element units per row (n % 4 == 0) and a row pointer aligned to one unit
static bool unit_aligned(const void* p, int bf16) { return (reinterpret_cast<uintptr_t>(p) & (bf16 ? 7u : 15u)) == 0; }

template <class T>
static int stack_split(const float* in, float* blocks, int64_t R, int64_t D, int64_t G, int64_t n_out, cudaStream_t stream)
{
    const int vec = (n_out % 4 == 0) && unit_aligned(in, !std::is_same_v<T, float>);
    stack_split_kernel<T><<<grid_for(G * R * (D / 4)), 256, 0, stream>>>(reinterpret_cast<const T*>(in), reinterpret_cast<typename Lanes<T>::V*>(blocks),
                                                                         R, static_cast<int>(D / 4), G, n_out, vec);
    return check_launch("stack_split_kernel");
}

template <class T>
static int stack_concat(const float* blocks, float* out, int64_t R, int64_t D, int64_t G, int64_t n_out, cudaStream_t stream)
{
    const int vec = (n_out % 4 == 0) && unit_aligned(out, !std::is_same_v<T, float>);
    stack_concat_kernel<T><<<grid_for(G * R * (D / 4)), 256, 0, stream>>>(reinterpret_cast<const typename Lanes<T>::V*>(blocks),
                                                                          reinterpret_cast<T*>(out), R, static_cast<int>(D / 4), G, n_out, vec);
    return check_launch("stack_concat_kernel");
}

template <class T>
static int stack_sum(const float* dxb, float* dx, int64_t R, int64_t D, int64_t G, int64_t n_in, cudaStream_t stream)
{
    const int vec = (n_in % 4 == 0) && unit_aligned(dx, !std::is_same_v<T, float>);
    stack_sum_kernel<T><<<grid_for(R * (D / 4)), 256, 0, stream>>>(reinterpret_cast<const float4*>(dxb), reinterpret_cast<T*>(dx), R,
                                                                    static_cast<int>(D / 4), G, n_in, vec);
    return check_launch("stack_sum_kernel");
}

int launch_stack_split(const float* in, float* blocks, int64_t R, int64_t D, int64_t G, int64_t n_out, cudaStream_t stream, int bf16)
{
    return bf16 ? stack_split<__nv_bfloat16>(in, blocks, R, D, G, n_out, stream) : stack_split<float>(in, blocks, R, D, G, n_out, stream);
}

int launch_stack_concat(const float* blocks, float* out, int64_t R, int64_t D, int64_t G, int64_t n_out, cudaStream_t stream, int bf16)
{
    return bf16 ? stack_concat<__nv_bfloat16>(blocks, out, R, D, G, n_out, stream) : stack_concat<float>(blocks, out, R, D, G, n_out, stream);
}

int launch_stack_sum(const float* dxb, float* dx, int64_t R, int64_t D, int64_t G, int64_t n_in, cudaStream_t stream, int bf16)
{
    return bf16 ? stack_sum<__nv_bfloat16>(dxb, dx, R, D, G, n_in, stream) : stack_sum<float>(dxb, dx, R, D, G, n_in, stream);
}

}  // namespace whvi
