// Device-side FWHT engine: register-resident butterflies + swizzled shared-memory
// transpositions between the views of layout.cuh.  sm_100a only.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <type_traits>
#include "layout.cuh"

namespace whvi {

// ---- compile-time loop -------------------------------------------------------------
template <int I, int End, class F>
__device__ __forceinline__ void static_for(F&& f)
{
    if constexpr (I < End) {
        f(std::integral_constant<int, I>{});
        static_for<I + 1, End>(f);
    }
}

enum ViewId : int { V_FIRST = 0, V_MID = 1, V_LAST = 2, V_MID2 = 3, V_NONE = 7 };

constexpr View get_view(int n, int c, int id)
{
    return id == V_FIRST ? view_first(n, c)
         : id == V_MID   ? view_mid(n, c)
         : id == V_LAST  ? view_last(n, c)
                         : view_mid2(n, c);
}

// A transform is a sequence of up to three view ids, packed 3 bits each (first = low).
constexpr int seq_pack(int a, int b = V_NONE, int c = V_NONE) { return a | (b << 3) | (c << 6); }
constexpr int seq_at(int seq, int i) { return (seq >> (3 * i)) & 7; }

// Is logical bit b (< k) butterflied in round `round` of sequence `seq`?
constexpr bool seq_bit_new(int n, int c, int k, int seq, int round, int b)
{
    if (b >= k) return false;
    for (int r = 0; r < round; ++r) {
        const View v = get_view(n, c, seq_at(seq, r));
        if (view_has(v, c, b)) return false;
    }
    const View v = get_view(n, c, seq_at(seq, round));
    return view_has(v, c, b);
}

// Same, ignoring the transform length (for kernels that take K at run time).
constexpr bool seq_bit_first_seen(int n, int c, int seq, int round, int b)
{
    for (int r = 0; r < round; ++r) {
        const View v = get_view(n, c, seq_at(seq, r));
        if (view_has(v, c, b)) return false;
    }
    const View v = get_view(n, c, seq_at(seq, round));
    return view_has(v, c, b);
}

// ---- memory helpers ------------------------------------------------------------------
__device__ __forceinline__ float4 ldg_stream(const float* p)
{
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ void stg_stream(float* p, const float4& v)
{
    asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z),
                 "f"(v.w)
                 : "memory");
}

// ---- activation I/O types (SURVEY 8f N4): fp32, or bf16 in HBM with fp32 arithmetic in registers ----------------------
// Io<T>::ld4 / st4 move four consecutive elements (16 bytes of fp32, 8 bytes of bf16) with the streaming cache hints.
template <class T>
struct Io;
template <>
struct Io<float> {
    static __device__ __forceinline__ float4 ld4(const float* p) { return ldg_stream(p); }
    static __device__ __forceinline__ void st4(float* p, const float4& v) { stg_stream(p, v); }
    // shared-memory side (bulk-copy staged tiles): read four elements widened to fp32, zero four elements
    static __device__ __forceinline__ float4 lds4(const float* p) { return *reinterpret_cast<const float4*>(p); }
    static __device__ __forceinline__ void sts_zero4(float* p) { *reinterpret_cast<float4*>(p) = make_float4(0.f, 0.f, 0.f, 0.f); }
};
template <>
struct Io<__nv_bfloat16> {
    static __device__ __forceinline__ float4 ld4(const __nv_bfloat16* p)
    {
        uint32_t a, b;
        asm volatile("ld.global.nc.L1::no_allocate.v2.b32 {%0,%1}, [%2];" : "=r"(a), "=r"(b) : "l"(p));
        // bf16 -> fp32 is exact: the 16 bits are the top half of the fp32 pattern
        return make_float4(__uint_as_float(a << 16), __uint_as_float(a & 0xFFFF0000u), __uint_as_float(b << 16), __uint_as_float(b & 0xFFFF0000u));
    }
    static __device__ __forceinline__ void st4(__nv_bfloat16* p, const float4& v)
    {
        uint32_t a, b;   // round to nearest even, two at a time (the first source operand lands in the upper half)
        asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(a) : "f"(v.y), "f"(v.x));
        asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(b) : "f"(v.w), "f"(v.z));
        asm volatile("st.global.L1::no_allocate.v2.b32 [%0], {%1,%2};" ::"l"(p), "r"(a), "r"(b) : "memory");
    }
    static __device__ __forceinline__ float4 lds4(const __nv_bfloat16* p)
    {
        const uint2 u = *reinterpret_cast<const uint2*>(p);
        return make_float4(__uint_as_float(u.x << 16), __uint_as_float(u.x & 0xFFFF0000u), __uint_as_float(u.y << 16),
                           __uint_as_float(u.y & 0xFFFF0000u));
    }
    static __device__ __forceinline__ void sts_zero4(__nv_bfloat16* p) { *reinterpret_cast<uint2*>(p) = make_uint2(0u, 0u); }
};

// Barrier among the T threads of one tile group.
template <int T, int GROUPS>
__device__ __forceinline__ void group_sync(int group)
{
    if constexpr (T == 32) {
        __syncwarp();
    } else if constexpr (GROUPS == 1) {
        __syncthreads();
    } else {
        asm volatile("bar.sync %0, %1;" ::"r"(group + 1), "n"(T) : "memory");
    }
}

// Barrier among T threads on named barrier `id` (T == 32: the threads are one warp).
template <int T>
__device__ __forceinline__ void role_sync(int id)
{
    if constexpr (T == 32) {
        __syncwarp();
    } else {
        asm volatile("bar.sync %0, %1;" ::"r"(id), "n"(T) : "memory");
    }
}
// Producer/consumer handshake between two thread sets on named barrier `id` (COUNT =
// total threads of both sets): the producer side arrives, the consumer side waits.
template <int COUNT>
__device__ __forceinline__ void bar_arrive(int id)
{
    asm volatile("bar.arrive %0, %1;" ::"r"(id), "n"(COUNT) : "memory");
}
template <int COUNT>
__device__ __forceinline__ void bar_wait(int id)
{
    asm volatile("bar.sync %0, %1;" ::"r"(id), "n"(COUNT) : "memory");
}
// Ask the L2 to fetch `bytes` (multiple of 16) starting at p (16-byte aligned).
__device__ __forceinline__ void l2_prefetch_bulk(const void* p, uint32_t bytes)
{
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}

// ---- mbarrier + bulk async copy (TMA, non-tensor form) ----------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    uint32_t done;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    } while (!done);
}
// global -> shared bulk copy (bytes: multiple of 16; both addresses 16-byte aligned); completion
// is signalled on `bar` as `bytes` of transaction count.
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// ---- butterflies -----------------------------------------------------------------------
// One radix-2 stage on register bit P.  For P >= 1 the two halves of each butterfly are
// handled as packed fp32x2 (FADD2 on sm_100a): the same IEEE fp32 adds, half the issue
// slots.
template <int E, int P>
__device__ __forceinline__ void bfly_stage(float (&v)[E])
{
    if constexpr (P == 0) {
#pragma unroll
        for (int r = 0; r < E; r += 2) {
            const float a = v[r], b = v[r + 1];
            v[r] = a + b;
            v[r + 1] = a - b;
        }
    } else {
#pragma unroll
        for (int r = 0; r < E; r += 2) {
            if (r & (1 << P)) continue;
            const float2 a = make_float2(v[r], v[r + 1]);
            const float2 b = make_float2(v[r + (1 << P)], v[r + (1 << P) + 1]);
            const float2 s = __fadd2_rn(a, b);
            const float2 d = __fadd2_rn(a, make_float2(-b.x, -b.y));
            v[r] = s.x;
            v[r + 1] = s.y;
            v[r + (1 << P)] = d.x;
            v[r + (1 << P) + 1] = d.y;
        }
    }
}

// Transform length as a template argument: KT >= 0 is log2(D) itself; KT < 0 encodes a
// run-time length k in the closed range [lo, hi] as KT = -(32*lo + hi) (one instantiation
// then serves a family of D; only stages on bits lo..hi-1 carry a uniform run-time guard).
constexpr int k_family(int lo, int hi) { return -(32 * lo + hi); }
constexpr int k_lo(int KT) { return KT >= 0 ? KT : (-KT) / 32; }
constexpr int k_hi(int KT) { return KT >= 0 ? KT : (-KT) % 32; }

// All butterflies of round ROUND of sequence SEQ for a transform over logical bits [0,k).
template <int N, int C, int KT, int SEQ, int ROUND>
__device__ __forceinline__ void bfly_round(float (&v)[1 << C], int k = KT)
{
    static_for<0, C>([&](auto p_) {
        constexpr int p = decltype(p_)::value;
        constexpr int b = get_view(N, C, seq_at(SEQ, ROUND)).bit[p];
        if constexpr (seq_bit_first_seen(N, C, SEQ, ROUND, b)) {
            if constexpr (b < k_lo(KT)) {
                bfly_stage<(1 << C), p>(v);
            } else if constexpr (b < k_hi(KT)) {
                if (b < k) bfly_stage<(1 << C), p>(v);
            }
        }
    });
}

// ---- transposition through shared memory -----------------------------------------------
// Writer side: thread `tid` holds v[] in view A; store every element at its physical
// address in the layout owned by reader view B.  phys = phys(tid part) ^ phys(reg part);
// the register part is a compile-time constant whose only bits overlapping the thread
// part are the swizzle bits [4:2].
template <int N, int C, int VA, int VB>
__device__ __forceinline__ uint32_t transpose_writer_base(uint32_t tid)
{
    uint32_t base = 0;
    static_for<0, N - C>([&](auto j_) {
        constexpr int j = decltype(j_)::value;
        constexpr View a = get_view(N, C, VA);
        constexpr View b = get_view(N, C, VB);
        constexpr uint32_t col = view_phys(b, 1u << a.bit[C + j]);
#if WHVI_PADDED
        base += ((tid >> j) & 1u) ? col : 0u;   // the padded map is additive over disjoint index bits
#else
        base ^= ((tid >> j) & 1u) ? col : 0u;
#endif
    });
    return base;
}

template <int N, int C, int VA, int VB>
__device__ __forceinline__ void transpose_write(const float (&v)[1 << C], float* buf, uint32_t wbase)
{
    static_for<0, (1 << C)>([&](auto r_) {
        constexpr int r = decltype(r_)::value;
        constexpr View a = get_view(N, C, VA);
        constexpr View b = get_view(N, C, VB);
        constexpr uint32_t pr = view_phys(b, view_reg_logical(a, r));
#if WHVI_PADDED
        buf[wbase + pr] = v[r];
#else
        constexpr uint32_t lo = pr & 0x1Cu;   // may overlap thread bits (swizzle): XOR
        constexpr uint32_t hi = pr & ~0x1Cu;  // disjoint from thread bits: additive
        buf[(wbase ^ lo) + hi] = v[r];
#endif
    });
}

// Reader side: thread `tid` (in view B) reads its E words as swizzled float4 slots.
template <int C>
__device__ __forceinline__ void transpose_read(float (&v)[1 << C], const float* buf, uint32_t tid)
{
    constexpr int E = 1 << C;
#if WHVI_PADDED
    const float* base = buf + tid * (E + 4);
#else
    const uint32_t sw = swz_of_tid(C, tid);
    const float* base = buf + (tid << C);
#endif
#pragma unroll
    for (int j = 0; j < E / 4; ++j) {
#if WHVI_PADDED
        const float4 q = *reinterpret_cast<const float4*>(base + 4 * j);
#else
        const float4 q = *reinterpret_cast<const float4*>(base + ((j ^ sw) << 2));
#endif
        v[4 * j + 0] = q.x;
        v[4 * j + 1] = q.y;
        v[4 * j + 2] = q.z;
        v[4 * j + 3] = q.w;
    }
}

// ---- global <-> registers in a FIRST/LAST-type view --------------------------------------
// Element offset (in floats, relative to the tile base) of this thread's float4 number m.
template <int N, int C, int V>
__device__ __forceinline__ uint32_t tile_thread_offset(uint32_t tid)
{
    constexpr View v = get_view(N, C, V);
    static_assert(v.bit[0] == 0 && v.bit[1] == 1, "view is not float4-addressable");
    uint32_t off = 0;
    static_for<0, N - C>([&](auto j_) {
        constexpr int j = decltype(j_)::value;
        constexpr int b = get_view(N, C, V).bit[C + j];
        off |= ((tid >> j) & 1u) << b;
    });
    return off;
}
template <int N, int C, int V>
constexpr uint32_t tile_reg_offset(int m)  // m = float4 index 0..E/4-1
{
    return view_reg_logical(get_view(N, C, V), static_cast<uint32_t>(m) << 2);
}

}  // namespace whvi
