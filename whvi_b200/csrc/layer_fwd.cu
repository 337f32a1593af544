// Kernel (2) [this file] and kernel (3) [layer_bwd.cu]: the fused WHVILinear forward and backward (PAPER semantics,
// docstring src/weights.py:77:  W = S1 H diag(g) H S2).
//
//   forward, per row (s,b):   y = s1 * H( g_s * H( s2 * x ) ) (+ bias)
//   backward (SURVEY App. A): dt3 = H(s1*dy);  dg_s = sum_b dt3 * t2;  dt1 = H(g_s*dt3)
//                             dx = s2*dt1;  ds2 = sum dt1*x;  ds1 = sum dy*t4;  dbias = sum dy
//                             with t2 = H(s2*x), t4 = H(g_s*t2) recomputed, nothing saved.
//
// The reference materialises W (D x D) through four FWHTs of D x D matrices and a dense
// GEMM per MC sample (src/weights.py:73, :93); here every activation row goes through HBM
// once per pass: 8 B/elt forward, 12 B/elt backward (read x, dy; write dx).
//
// Structure: a tile (one row, or N/D rows when D < N) is held in registers by T threads,
// E floats each; H is the register/shared-memory engine of engine.cuh (views FIRST -> MID
// -> LAST on the way in, LAST -> MID2 -> FIRST on the way out), so x, y, dy, dx, s1, s2 and
// g are all touched as coalesced float4s.

#include "layer_common.cuh"

namespace whvi {

struct FwdArgs {
    const float* x;
    int64_t x_sample_stride;
    const float* g;
    const float* s1;
    const float* s2;
    const float* bias;
    float* y;
    int64_t sample_elems;  // B * D
    int n_samples;          // S
    int ctas_per_sample;
    int iters_per_group;
    int k;                  // log2(D)
    int relu_out;           // y = max(y, 0)
    // FROM_T2: x already holds t2 = H(s2 * x) (sample-independent by linearity, SURVEY 8d C5:
    // computed once per input row with whvi_fwht_f32), so one transform per (sample, row) is left
    const float* target;    // HAS_TARGET: (B, D); sum (y - target)^2 goes to sq_partials[cta]
    float* sq_partials;
    int spg;                // grouped launch: samples per parameter group (n_samples when there is one group)
    int pstride, bstride;   // floats between consecutive groups' s1 / s2 vectors, bias vectors
};

// ------------------------------------------------------------------------------ forward
// ROUNDS == 3: FIRST -> MID -> LAST, g applied in LAST (global float4 reads), LAST -> MID2 -> FIRST.
// ROUNDS == 2: FIRST -> MID, g applied in MID from the shared-memory table, MID -> FIRST.
// BUFS: tile buffers per group (2 = ping-pong, 1 = in place with one more barrier per
// transposition but half the shared memory).
// Flags that guard LOADS are template parameters: a run-time branch around a load inside the
// unrolled float4 loops stops the compiler from batching the loads (measured: 2x slower).
// IO: the activations' type in HBM (float, or __nv_bfloat16 with fp32 arithmetic in registers: SURVEY 8f N4); a.x / a.y are
// then IO pointers behind the float* of FwdArgs.  Parameters, g and the target are always fp32.
template <int N, int C, int KT, int GROUPS, int ROUNDS, int BUFS, int MINB, bool HAS_BIAS, bool HAS_TARGET, bool FROM_T2, class IO = float>
__global__ void __launch_bounds__((1 << (N - C)) * GROUPS, MINB) layer_fwd_kernel(const FwdArgs a)
{
    constexpr int T = 1 << (N - C);
    constexpr int E = 1 << C;
    constexpr int64_t TILE = int64_t(1) << N;
    static_assert(ROUNDS == 3 || rounds_needed(N, C, N) <= 2, "2-view kernel needs FIRST+MID to cover all bits");
    static_assert(rounds_needed(N, C, N) <= 3, "FIRST+MID+LAST must cover every tile bit (e.g. 5+5+3 = 13 bits at C = 5)");
    extern __shared__ float4 smem4[];
    float* smem = reinterpret_cast<float*>(smem4);
    const int group = threadIdx.x / T;
    const uint32_t tid = threadIdx.x % T;
    const int bar = group + 1;
    const int k = KT >= 0 ? KT : a.k;
    const uint32_t cmask = (1u << k) - 1u;
    // sample-minor CTA order: the S CTAs working on the same tile range of different samples
    // are neighbours in launch order, so sample-independent operands (a shared x block, the
    // MNLL target) come from DRAM once and hit L2 for the other S-1 samples
    const int s = blockIdx.x % a.n_samples;
    const int cta_in_sample = blockIdx.x / a.n_samples;
    const float* __restrict__ gs = a.g + (int64_t(s) << k);
    const int grp = s / a.spg, sx = s - grp * a.spg;   // parameter group (Stacked block) and the sample whose input it reads
    const float* __restrict__ s1p = a.s1 + int64_t(grp) * a.pstride;
    const float* __restrict__ s2p = a.s2 + int64_t(grp) * a.pstride;
    const float* __restrict__ biasp = HAS_BIAS ? a.bias + int64_t(grp) * a.bstride : nullptr;
    constexpr size_t SW = scratch_words(N, C);  // one transposition buffer / g table (== TILE unless WHVI_PADDED)
    float* gt = smem;  // ROUNDS == 2 only
    float* bufA = smem + (ROUNDS == 2 ? SW : 0) + size_t(group) * BUFS * SW;
    float* bufB = bufA + (BUFS == 2 ? SW : 0);
    const float relu_floor = a.relu_out ? 0.f : -INFINITY;

    const uint32_t off_f = tile_thread_offset<N, C, V_FIRST>(tid);
    const uint32_t wb_fm = transpose_writer_base<N, C, V_FIRST, V_MID>(tid);
    uint32_t off_l = 0, wb_ml = 0, wb_lm = 0, wb_mf = 0, gbase = 0;
    if constexpr (ROUNDS == 3) {
        off_l = tile_thread_offset<N, C, V_LAST>(tid);
        wb_ml = transpose_writer_base<N, C, V_MID, V_LAST>(tid);
        wb_lm = transpose_writer_base<N, C, V_LAST, V_MID2>(tid);
        wb_mf = transpose_writer_base<N, C, V_MID2, V_FIRST>(tid);
    } else {
        wb_mf = transpose_writer_base<N, C, V_MID, V_FIRST>(tid);
        gbase = gtab_base<N, C>(tid, k);
        gtab_fill<N, C>(gt, gs, T * GROUPS, k);
        __syncthreads();
    }

    float sq = 0.f;
#pragma unroll 1
    for (int it = 0; it < a.iters_per_group; ++it) {
        const int64_t tile = (int64_t(cta_in_sample) * a.iters_per_group + it) * GROUPS + group;
        const int64_t e0 = tile * TILE;  // element offset inside the sample
        if (e0 >= a.sample_elems) break;  // uniform per group
        const int64_t left = a.sample_elems - e0;
        const IO* __restrict__ xs = reinterpret_cast<const IO*>(a.x) + int64_t(sx) * a.x_sample_stride + e0;
        IO* __restrict__ ys = reinterpret_cast<IO*>(a.y) + int64_t(s) * a.sample_elems + e0;
        if (tid == 0 && it + 1 < a.iters_per_group) {  // pull the group's next tile towards L2
            const int64_t e1 = e0 + GROUPS * TILE;
            if (e1 < a.sample_elems) {
                const int64_t left1 = a.sample_elems - e1;
                const uint32_t bytes = static_cast<uint32_t>((left1 < TILE ? left1 : TILE) * sizeof(IO));
                if constexpr (sizeof(IO) < sizeof(float)) {
                    // a bulk prefetch takes a 16-byte-aligned address and whole 16-byte units; a bf16 sample of B * D % 8 != 0
                    // elements (D = 4 with an odd B) starts 8 bytes off and ends on half a unit: prefetch the whole units
                    // of aligned tiles only
                    const bool aligned = (reinterpret_cast<uintptr_t>(xs + GROUPS * TILE) & 15u) == 0;
                    if (aligned && bytes >= 16) l2_prefetch_bulk(xs + GROUPS * TILE, bytes & ~15u);
                } else {
                    l2_prefetch_bulk(xs + GROUPS * TILE, bytes);
                }
            }
        }

        float v[E];
        if constexpr (FROM_T2 && ROUNDS == 3) {
            // t2 read straight in the LAST view (also float4-coalesced), times g, then H
            for_each_vec<N, C, V_LAST>(off_l, cmask, [&](auto m_, uint32_t off, uint32_t coord) {
                constexpr int m = decltype(m_)::value;
                float4 q = make_float4(0.f, 0.f, 0.f, 0.f);
                if (off < left) q = Io<IO>::ld4(xs + off);
                const float4 w = ldg4(gs + coord);
                mul4(v + 4 * m, q, w);
            });
            transform_out<N, C, KT, T, BUFS == 1>(v, bufA, bufB, tid, bar, k, wb_lm, wb_mf);
        } else {
            for_each_vec<N, C, V_FIRST>(off_f, cmask, [&](auto m_, uint32_t off, uint32_t coord) {
                constexpr int m = decltype(m_)::value;
                float4 q = make_float4(0.f, 0.f, 0.f, 0.f);
                if (off < left) q = Io<IO>::ld4(xs + off);
                if constexpr (FROM_T2) {
                    v[4 * m] = q.x, v[4 * m + 1] = q.y, v[4 * m + 2] = q.z, v[4 * m + 3] = q.w;
                } else {
                    const float4 w = ldg4(s2p + coord);
                    mul4(v + 4 * m, q, w);
                }
            });
            if constexpr (ROUNDS == 3) {
                transform_in<N, C, KT, T, BUFS == 1>(v, bufA, bufB, tid, bar, k, wb_fm, wb_ml);
                for_each_vec<N, C, V_LAST>(off_l, cmask, [&](auto m_, uint32_t, uint32_t coord) {
                    constexpr int m = decltype(m_)::value;
                    const float4 w = ldg4(gs + coord);
                    scale4(v + 4 * m, w);
                });
                transform_out<N, C, KT, T, BUFS == 1>(v, bufA, bufB, tid, bar, k, wb_lm, wb_mf);
            } else {
                // FROM_T2: the first transform is already done; only the move to the MID view is left
                if constexpr (!FROM_T2) bfly_round<N, C, KT, SEQ2_IN, 0>(v, k);
                if constexpr (BUFS == 1) role_sync<T>(bar);  // previous tile's reads of bufA are done
                transpose_write<N, C, V_FIRST, V_MID>(v, bufA, wb_fm);
                role_sync<T>(bar);
                transpose_read<C>(v, bufA, tid);
                if constexpr (!FROM_T2) bfly_round<N, C, KT, SEQ2_IN, 1>(v, k);
                gtab_for_each<N, C>(gt, gbase, [&](auto j_, const float4 w) {
                    constexpr int j = decltype(j_)::value;
                    scale4(v + 4 * j, w);
                });
                bfly_round<N, C, KT, SEQ2_OUT, 0>(v, k);
                if constexpr (BUFS == 1) role_sync<T>(bar);
                transpose_write<N, C, V_MID, V_FIRST>(v, bufB, wb_mf);
                role_sync<T>(bar);
                transpose_read<C>(v, bufB, tid);
                bfly_round<N, C, KT, SEQ2_OUT, 1>(v, k);
            }
        }
        for_each_vec<N, C, V_FIRST>(off_f, cmask, [&](auto m_, uint32_t off, uint32_t coord) {
            constexpr int m = decltype(m_)::value;
            const float4 w = ldg4(s1p + coord);
            float4 o = make_float4(v[4 * m] * w.x, v[4 * m + 1] * w.y, v[4 * m + 2] * w.z, v[4 * m + 3] * w.w);
            if constexpr (HAS_BIAS) {
                const float4 b = ldg4(biasp + coord);
                o.x += b.x;
                o.y += b.y;
                o.z += b.z;
                o.w += b.w;
            }
            o.x = fmaxf(o.x, relu_floor);
            o.y = fmaxf(o.y, relu_floor);
            o.z = fmaxf(o.z, relu_floor);
            o.w = fmaxf(o.w, relu_floor);
            if (off < left) {
                if constexpr (HAS_TARGET) {
                    // streaming load: the target must not evict s1/s2 from the small L1 that is
                    // left next to 192 KB of shared memory
                    const float4 tg = ldg_stream(a.target + e0 + off);
                    const float d0 = o.x - tg.x, d1 = o.y - tg.y, d2 = o.z - tg.z, d3 = o.w - tg.w;
                    sq = fmaf(d0, d0, fmaf(d1, d1, fmaf(d2, d2, fmaf(d3, d3, sq))));
                }
                Io<IO>::st4(ys + off, o);
            }
        });
    }

    if constexpr (HAS_TARGET) {  // fixed-order CTA reduction of the squared residuals
        __shared__ float red[32];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = sq;
        __syncthreads();
        if (threadIdx.x == 0) {
            float tot = 0.f;
            for (int w = 0; w < (T * GROUPS) / 32; ++w) tot += red[w];
            a.sq_partials[blockIdx.x] = tot;
        }
    }
}

template <int N, int C, int KT, int GROUPS, int ROUNDS, int BUFS, int MINB>
static int launch_fwd_cfg(const LayerFwdCall& c, int k, cudaStream_t stream)
{
    static unsigned char smem_ok[10][64] = {};
    constexpr int threads = (1 << (N - C)) * GROUPS;
    constexpr size_t tile = size_t(1) << N;
    constexpr size_t sw = scratch_words(N, C);
    constexpr size_t smem = sizeof(float) * (sw * BUFS * GROUPS + (ROUNDS == 2 ? sw : 0));
    const int64_t D = int64_t(1) << k;
    const int64_t tiles_per_sample = (c.B * D + int64_t(tile) - 1) / int64_t(tile);
    // persistent CTAs: 2-view kernels amortise the g-table fill over >= 4 tiles per group, and
    // every kernel prefetches its group's next tile into L2 while it works on the current one
    const Plan plan = make_plan(c.S, tiles_per_sample, GROUPS, 148 * 16, ROUNDS == 2 ? 4 : 2);
    const int64_t ctas = int64_t(plan.ctas_per_sample) * c.S;
    if (c.partials_needed) {
        *c.partials_needed = static_cast<size_t>(ctas);
        return WHVI_OK;
    }
    if (ctas > 0x7fffffffLL) return fail(WHVI_E_SHAPE, "layer_fwd: grid too large");
    FwdArgs a{c.x, c.xs, c.g, c.s1, c.s2, c.bias, c.y, c.B * D, static_cast<int>(c.S), plan.ctas_per_sample, plan.iters_per_group, k,
              c.relu_out, c.target, c.sq_partials, static_cast<int>(c.S / c.groups), static_cast<int>(c.pstride), static_cast<int>(c.bstride)};
    auto go = [&](auto kernel, int slot) -> int {
        if (int rc = ensure_smem(kernel, smem, smem_ok[slot])) return rc;
        kernel<<<static_cast<unsigned>(ctas), threads, smem, stream>>>(a);
        return check_launch("layer_fwd_kernel");
    };
    const bool hb = c.bias != nullptr, ht = c.target != nullptr;
    if (c.bf16) {   // bf16 activations in HBM (inference paths: no target)
        if (ht) return fail(WHVI_E_MODE, "layer_fwd: bf16 activations cannot be combined with a target");
        if (c.from_t2) {
            if (hb) return go(layer_fwd_kernel<N, C, KT, GROUPS, ROUNDS, BUFS, MINB, true, false, true, __nv_bfloat16>, 6);
            return go(layer_fwd_kernel<N, C, KT, GROUPS, ROUNDS, BUFS, MINB, false, false, true, __nv_bfloat16>, 7);
        }
        if (hb) return go(layer_fwd_kernel<N, C, KT, GROUPS, ROUNDS, BUFS, MINB, true, false, false, __nv_bfloat16>, 8);
        return go(layer_fwd_kernel<N, C, KT, GROUPS, ROUNDS, BUFS, MINB, false, false, false, __nv_bfloat16>, 9);
    }
    if (c.from_t2) {
        if (ht) return fail(WHVI_E_MODE, "layer_fwd: FROM_T2 cannot be combined with a target");
        if (hb) return go(layer_fwd_kernel<N, C, KT, GROUPS, ROUNDS, BUFS, MINB, true, false, true>, 4);
        return go(layer_fwd_kernel<N, C, KT, GROUPS, ROUNDS, BUFS, MINB, false, false, true>, 5);
    }
    if (hb && ht) return go(layer_fwd_kernel<N, C, KT, GROUPS, ROUNDS, BUFS, MINB, true, true, false>, 0);
    if (hb) return go(layer_fwd_kernel<N, C, KT, GROUPS, ROUNDS, BUFS, MINB, true, false, false>, 1);
    if (ht) return go(layer_fwd_kernel<N, C, KT, GROUPS, ROUNDS, BUFS, MINB, false, true, false>, 2);
    return go(layer_fwd_kernel<N, C, KT, GROUPS, ROUNDS, BUFS, MINB, false, false, false>, 3);
}

int launch_layer_fwd(const LayerFwdCall& c, int64_t D, cudaStream_t stream)
{
    const int k = ilog2(D);
    // D <= 64: three views (the middle multiply reads g from global memory)
    if (k >= 2 && k <= 6) return launch_fwd_cfg<10, 5, k_family(2, 6), 4, 3, 2, 4>(c, k, stream);
    // 128 <= D <= 1024: two views, one warp per 1024-float tile (exact-K code for D = 1024:
    // the run-time guards of a family cost ~8% there)
    if (k >= 7 && k <= 9) return launch_fwd_cfg<10, 5, k_family(7, 9), 8, 2, 2, 3>(c, k, stream);
    if (k == 10) return launch_fwd_cfg<10, 5, 10, 8, 2, 2, 3>(c, k, stream);
    // D = 2048, 4096: two views with 64 floats per thread (tile = 4096 = one or two rows)
    if (k == 11) return launch_fwd_cfg<12, 6, 11, 2, 2, 1, 4>(c, k, stream);
    if (k == 12) return launch_fwd_cfg<12, 6, 12, 2, 2, 1, 4>(c, k, stream);
    // D = 8192: three views, 32 floats per thread
    // D = 8192: three views, 64 floats per thread, one in-place buffer, 4 CTAs of 128 threads per
    // SM (measured 68% of the HBM roofline vs 60% for 32 floats/thread with ping-pong buffers; two 4096-float halves
    // through the two-view engine with the other half in tensor memory measured 62%, profiles/r02_fwd_split_8192.md)
    if (k == 13) return launch_fwd_cfg<13, 6, 13, 1, 3, 1, 4>(c, k, stream);
    // D = 16384, 32768 (forward only: MC predictive evaluation, BASELINE config 5): three views,
    // 64 floats per thread, one in-place transposition buffer (64 / 128 KB)
    if (k == 14) return launch_fwd_cfg<14, 6, 14, 1, 3, 1, 2>(c, k, stream);   // two 64 KB CTAs per SM: 128 registers per thread (one CTA at 218 registers ran at 35% of the roofline)
    if (k == 15) return launch_fwd_cfg<15, 6, 15, 1, 3, 1, 1>(c, k, stream);
    return fail(WHVI_E_SHAPE, "layer_fwd: D = %lld unsupported (4 <= D <= 32768)", (long long)D);
}

}  // namespace whvi
