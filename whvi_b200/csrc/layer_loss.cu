// Fused LAST layer of a regression network: WHVILinear forward + Gaussian-MNLL residual +
// WHVILinear backward in ONE pass over the layer's input (SURVEY 8f N1 taken to its end).
//
//   y_hat = s1 * H(g * H(s2 * x)) (+ bias)          never written to HBM
//   r     = y_hat - target                          sum r^2 -> the MNLL data term (src/likelihoods.py:18-29)
//   dy    = r   (unit loss coefficient; the caller scales by 2 * dMNLL/dsq afterwards)
//   dx, dg, ds1, ds2, dbias as in layer_bwd.cu
//
// Separate forward + backward kernels move 8 + 12 = 20 B/elt for this layer (x in, y_hat out;
// y_hat, x in, dx out) and the backward recomputes the forward's two transforms anyway; fused,
// the layer costs the backward's four transforms and 8 B/elt (x in, dx out; the target is shared
// by all samples and stays in L2).
//
// Structure: the TMA-staged two-role kernel of layer_bwd.cu, but the roles are pipelined instead
// of symmetric.  For every tile
//   X role:  t2 = H(s2*x) -> publishes t2 -> t4 = H(g*t2) -> y_hat, r, sum r^2, ds1 += r*t4,
//            dbias += r -> publishes r in the stage's second tile
//   Y role:  (one half-tile behind) dt3 = H(s1*r) -> dg += dt3*t2 -> dt1 = H(g*dt3) -> ds2 += dt1*x,
//            dx = s2*dt1 (masked by x > 0 after a fused ReLU)
// Stage = [x tile | target tile]; both arrive by bulk async copy and X overwrites the target tile
// in place with r.  mbarriers per stage: full (TMA landed), ready (X -> Y: r and t2 published),
// empty (Y -> producer).  Because Y works one tile behind X, the ring is NS = 3 deep and the
// producer (thread 0 of X) refills a stage at the END of its iteration: the stage it needs was
// released by Y one tile ago, so it does not stall, and the copy still has a whole tile of lead
// time.  (With 2 stages and the refill at the start of an iteration X waits for Y and the two
// roles serialise: measured 2x slower.)
// The transposition buffers of THIS translation unit use the padded (XOR-free) layout (WHVI_PADDED_BWD, default 1;
// measured: the backward gains ~4% at D = 1024...8192 with bit-identical outputs, the two-view forward does not,
// profiles/r01_bwd_notes.md item 14, profiles/r02_ab_padbwd.txt); -DWHVI_PADDED_BWD=0 builds the swizzled variant.
#ifndef WHVI_PADDED_BWD
#define WHVI_PADDED_BWD 1   // product default since round 2: bit-identical outputs, -4% (profiles/r02_ab_padbwd.txt)
#endif
#if WHVI_PADDED_BWD && !defined(WHVI_PADDED)
#define WHVI_PADDED 1
#endif
#include "layer_common.cuh"

namespace whvi {


// IO: the type of x and dx in HBM (see layer_bwd_tma_kernel): a bf16 x tile is staged in the first half of its fp32-sized
// slot and widened on every read, dx is rounded once at the store; the target ring, r, t2 and all arithmetic stay fp32.
template <int N, int C, int KT, int PAIRS, int NS, bool SINGLE, int PREG, int ROUNDS, bool HAS_BIAS, class IO = float>
__global__ void __launch_bounds__((2 << (N - C)) * PAIRS, 1) layer_loss_kernel(const LossArgs p)
{
    constexpr int T = 1 << (N - C);
    constexpr int E = 1 << C;
    constexpr int64_t TILE = int64_t(1) << N;
    constexpr int SCR = SINGLE ? 1 : 2;
    constexpr int SW = int(scratch_words(N, C));  // one transposition buffer (== TILE unless WHVI_PADDED)
    constexpr int PAIR_FLOATS = WHVI_PADDED ? (2 * NS + NS) * int(TILE) + 2 * SCR * SW
                                            : (2 * NS + 2 * SCR + NS) * int(TILE);  // stages, scratch, one full t2 stash per stage
    static_assert(ROUNDS == 3 || rounds_needed(N, C, N) <= 2, "2-view kernel needs FIRST+MID to cover all bits");
    static_assert(rounds_needed(N, C, N) <= 3, "FIRST+MID+LAST must cover every tile bit");
    static_assert(ROUNDS == 3 || PREG > 0, "the 2-view loss kernel keeps g in registers");
    extern __shared__ float4 smem4[];
    __shared__ uint64_t full_bar[PAIRS][NS], empty_bar[PAIRS][NS], ready_bar[PAIRS][NS];
    float* smem = reinterpret_cast<float*>(smem4);
    const int k = KT >= 0 ? KT : p.k;
    const uint32_t cmask = (1u << k) - 1u;
    const int s = blockIdx.x % p.n_samples;  // sample-minor CTA order: the target tile is reused out of L2
    const int cta_in_sample = blockIdx.x / p.n_samples;
    const IO* __restrict__ xbase = reinterpret_cast<const IO*>(p.x) + int64_t(s) * p.x_sample_stride;

    if (threadIdx.x == 0) {
        for (int q = 0; q < PAIRS; ++q)
            for (int st = 0; st < NS; ++st) {
                mbar_init(&full_bar[q][st], 1);
                mbar_init(&empty_bar[q][st], T);   // the Y role releases a stage
                mbar_init(&ready_bar[q][st], T);   // the X role publishes r and t2
            }
        mbar_fence_init();
    }
    __syncthreads();

    auto tile_of = [&](int it, int pr) -> int64_t {
        return ((int64_t(cta_in_sample) * p.iters_per_group + it) * PAIRS + pr) * TILE;
    };
    auto issue_tile = [&](int it, int pr) {  // in-band producer (thread 0 of the X role), see layer_bwd.cu
        if (it >= p.iters_per_group) return;
        const int64_t e0 = tile_of(it, pr);
        if (e0 >= p.sample_elems) return;
        const int st = it % NS;
        if (it >= NS) mbar_wait(&empty_bar[pr][st], ((it / NS) & 1) ^ 1);
        const int64_t left = p.sample_elems - e0;
        const int64_t n = left < TILE ? left : TILE;
        const uint32_t bytes = static_cast<uint32_t>(n * sizeof(float));
        float* stage = smem + size_t(pr) * PAIR_FLOATS + size_t(st) * 2 * TILE;
        if constexpr (std::is_same_v<IO, float>) {
            mbar_arrive_expect_tx(&full_bar[pr][st], 2 * bytes);
            bulk_g2s(stage, xbase + e0, bytes, &full_bar[pr][st]);
        } else {
            const uint32_t xbytes = static_cast<uint32_t>(n * sizeof(IO));
            mbar_arrive_expect_tx(&full_bar[pr][st], xbytes + bytes);
            bulk_g2s(stage, xbase + e0, xbytes, &full_bar[pr][st]);
        }
        bulk_g2s(stage + TILE, p.target + e0, bytes, &full_bar[pr][st]);
    };

    const int role = threadIdx.x / (T * PAIRS);        // 0 = X, 1 = Y (warp-uniform)
    const int pair = (threadIdx.x % (T * PAIRS)) / T;
    const uint32_t tid = threadIdx.x % T;
    float* pair_smem = smem + size_t(pair) * PAIR_FLOATS;
#if WHVI_PADDED
    float* scratch = pair_smem + (2 * NS) * TILE + (SCR * role) * SW;
    float* scratch2 = scratch + (SINGLE ? 0 : SW);
    float* stash0 = pair_smem + (2 * NS) * TILE + 2 * SCR * SW;       // + st * TILE
#else
    float* scratch = pair_smem + (2 * NS + SCR * role) * TILE;
    float* scratch2 = scratch + (SINGLE ? 0 : TILE);
    float* stash0 = pair_smem + (2 * NS + 2 * SCR) * TILE;       // + st * TILE
#endif
    const int bar_role = 1 + 2 * pair + role;
    const float* __restrict__ gs = p.g + (int64_t(s) << k);
    const float relu_thr = p.relu_in ? 0.f : -INFINITY;

    const uint32_t off_f = tile_thread_offset<N, C, V_FIRST>(tid);
    const uint32_t off_l = tile_thread_offset<N, C, V_LAST>(tid);
    const uint32_t wb_fm = transpose_writer_base<N, C, V_FIRST, V_MID>(tid);
    const uint32_t wb_ml = transpose_writer_base<N, C, V_MID, V_LAST>(tid);
    const uint32_t wb_lm = transpose_writer_base<N, C, V_LAST, V_MID2>(tid);
    const uint32_t wb_mf = ROUNDS == 3 ? transpose_writer_base<N, C, V_MID2, V_FIRST>(tid)
                                       : transpose_writer_base<N, C, V_MID, V_FIRST>(tid);
    const uint32_t mid_logical = view_tid_logical(view_mid(N, C), tid);
    const uint32_t st_base = tid << C;                 // this thread's E floats in a t2 stash
    const uint32_t st_swz = swz_of_tid(C, tid);
    const int64_t slab_index = (int64_t(s) * p.ctas_per_sample + cta_in_sample) * PAIRS + pair;
    float* __restrict__ slab = p.ws + slab_index * 4 * TILE;

    auto to_mid = [&](float (&v)[E]) {
        if constexpr (ROUNDS == 3) {
            transform_in<N, C, KT, T, SINGLE>(v, scratch, scratch2, tid, bar_role, k, wb_fm, wb_ml);
        } else {
            bfly_round<N, C, KT, SEQ2_IN, 0>(v, k);
            if constexpr (SINGLE) role_sync<T>(bar_role);
            transpose_write<N, C, V_FIRST, V_MID>(v, scratch, wb_fm);
            role_sync<T>(bar_role);
            transpose_read<C>(v, scratch, tid);
            bfly_round<N, C, KT, SEQ2_IN, 1>(v, k);
        }
    };
    auto from_mid = [&](float (&v)[E]) {
        if constexpr (ROUNDS == 3) {
            transform_out<N, C, KT, T, SINGLE>(v, scratch, scratch2, tid, bar_role, k, wb_lm, wb_mf);
        } else {
            bfly_round<N, C, KT, SEQ2_OUT, 0>(v, k);
            if constexpr (SINGLE) role_sync<T>(bar_role);
            transpose_write<N, C, V_MID, V_FIRST>(v, scratch2, wb_mf);
            role_sync<T>(bar_role);
            transpose_read<C>(v, scratch2, tid);
            bfly_round<N, C, KT, SEQ2_OUT, 1>(v, k);
        }
    };
    auto load_g_regs = [&](float* gr) {
        if constexpr (ROUNDS == 3) {
            for_each_vec<N, C, V_LAST>(off_l, cmask, [&](auto m_, uint32_t, uint32_t coord) {
                constexpr int m = decltype(m_)::value;
                const float4 w = ldg4(gs + coord);
                gr[4 * m] = w.x, gr[4 * m + 1] = w.y, gr[4 * m + 2] = w.z, gr[4 * m + 3] = w.w;
            });
        } else {
            static_for<0, E>([&](auto r_) {
                constexpr int r = decltype(r_)::value;
                constexpr uint32_t rl = view_reg_logical(view_mid(N, C), r);
                gr[r] = __ldg(gs + ((mid_logical | rl) & cmask));
            });
        }
    };
    auto apply_g = [&](float (&v)[E], const float* gr) {
        if constexpr (PREG > 0) {
#pragma unroll
            for (int m = 0; m < E / 4; ++m) scale4(v + 4 * m, make_float4(gr[4 * m], gr[4 * m + 1], gr[4 * m + 2], gr[4 * m + 3]));
        } else {
            for_each_vec<N, C, V_LAST>(off_l, cmask, [&](auto m_, uint32_t, uint32_t coord) {
                constexpr int m = decltype(m_)::value;
                scale4(v + 4 * m, ldg4(gs + coord));
            });
        }
    };
    auto load_first_regs = [&](const float* vec, float* dst) {
        for_each_vec<N, C, V_FIRST>(off_f, cmask, [&](auto m_, uint32_t, uint32_t coord) {
            constexpr int m = decltype(m_)::value;
            const float4 w = ldg4(vec + coord);
            dst[4 * m] = w.x, dst[4 * m + 1] = w.y, dst[4 * m + 2] = w.z, dst[4 * m + 3] = w.w;
        });
    };
    auto first_param = [&](const float* regs, const float* vec, int m, uint32_t coord, bool in_regs) -> float4 {
        return in_regs ? make_float4(regs[4 * m], regs[4 * m + 1], regs[4 * m + 2], regs[4 * m + 3]) : ldg4(vec + coord);
    };

    if (role == 0) {
        // ------------------------------------------------------------------ X role
        float s2r[PREG ? E : 1], s1r[PREG ? E : 1], gr[PREG ? E : 1];
        if constexpr (PREG > 0) {
            load_first_regs(p.s2, s2r);
            load_first_regs(p.s1, s1r);
            load_g_regs(gr);
        }
        float acc_1[E];
        float acc_b[HAS_BIAS ? E : 1];
        float sq = 0.f;
#pragma unroll
        for (int i = 0; i < E; ++i) acc_1[i] = 0.f;
        if constexpr (HAS_BIAS) {
#pragma unroll
            for (int i = 0; i < E; ++i) acc_b[i] = 0.f;
        }
        if (tid == 0)
            for (int i = 0; i < NS - 1; ++i) issue_tile(i, pair);
#pragma unroll 1
        for (int it = 0; it < p.iters_per_group; ++it) {
            const int64_t e0 = tile_of(it, pair);
            if (e0 >= p.sample_elems) break;
            const int64_t left = p.sample_elems - e0;
            const int st = it % NS;
            float* stage_x = pair_smem + size_t(st) * 2 * TILE;
            float* stage_t = stage_x + TILE;   // target on arrival ...
            float* stage_r = stage_t;          // ... overwritten in place with r
            float* stash = stash0 + size_t(st) * TILE;
            mbar_wait(&full_bar[pair][st], (it / NS) & 1);
            if (left < TILE) {  // partial tile: zero this thread's float4s beyond the valid part (x and target)
                static_for<0, E / 4>([&](auto m_) {
                    constexpr int m = decltype(m_)::value;
                    const uint32_t off = off_f + tile_reg_offset<N, C, V_FIRST>(m);
                    if (off >= left) {
                        Io<IO>::sts_zero4(reinterpret_cast<IO*>(stage_x) + off);
                        *reinterpret_cast<float4*>(stage_t + off) = make_float4(0.f, 0.f, 0.f, 0.f);
                    }
                });
            }
            float a[E];
            for_each_vec<N, C, V_FIRST>(off_f, cmask, [&](auto m_, uint32_t off, uint32_t coord) {
                constexpr int m = decltype(m_)::value;
                const float4 q = Io<IO>::lds4(reinterpret_cast<const IO*>(stage_x) + off);
                mul4(a + 4 * m, q, first_param(s2r, p.s2, m, coord, PREG > 0));
            });
            to_mid(a);  // a = t2
#pragma unroll
            for (int j = 0; j < E / 4; ++j)  // publish t2 (thread-private swizzled float4 slots)
                *reinterpret_cast<float4*>(stash + st_base + ((j ^ st_swz) << 2)) = make_float4(a[4 * j], a[4 * j + 1], a[4 * j + 2], a[4 * j + 3]);
            apply_g(a, gr);
            from_mid(a);  // a = t4 (FIRST layout)
            for_each_vec<N, C, V_FIRST>(off_f, cmask, [&](auto m_, uint32_t off, uint32_t coord) {
                constexpr int m = decltype(m_)::value;
                const float4 w = first_param(s1r, p.s1, m, coord, PREG > 0);
                float4 y = make_float4(a[4 * m] * w.x, a[4 * m + 1] * w.y, a[4 * m + 2] * w.z, a[4 * m + 3] * w.w);
                if constexpr (HAS_BIAS) {
                    const float4 bb = ldg4(p.bias + coord);
                    y.x += bb.x, y.y += bb.y, y.z += bb.z, y.w += bb.w;
                }
                const float4 tg = *reinterpret_cast<const float4*>(stage_t + off);
                const bool valid = left >= TILE || off < left;
                const float4 r = valid ? make_float4(y.x - tg.x, y.y - tg.y, y.z - tg.z, y.w - tg.w) : make_float4(0.f, 0.f, 0.f, 0.f);
                sq = fmaf(r.x, r.x, fmaf(r.y, r.y, fmaf(r.z, r.z, fmaf(r.w, r.w, sq))));
                fma4(acc_1 + 4 * m, r, a + 4 * m);
                if constexpr (HAS_BIAS) {
                    acc_b[4 * m] += r.x, acc_b[4 * m + 1] += r.y, acc_b[4 * m + 2] += r.z, acc_b[4 * m + 3] += r.w;
                }
                *reinterpret_cast<float4*>(stage_r + off) = r;  // the Y role's upstream gradient
            });
            mbar_arrive(&ready_bar[pair][st]);  // release: r and t2 of this tile are published
            if (tid == 0) issue_tile(it + NS - 1, pair);  // refill the stage Y released one tile ago
        }
        for_each_vec<N, C, V_FIRST>(off_f, cmask, [&](auto m_, uint32_t off, uint32_t) {
            constexpr int m = decltype(m_)::value;
            *reinterpret_cast<float4*>(slab + TILE + off) = make_float4(acc_1[4 * m], acc_1[4 * m + 1], acc_1[4 * m + 2], acc_1[4 * m + 3]);
            if constexpr (HAS_BIAS)
                *reinterpret_cast<float4*>(slab + 3 * TILE + off) = make_float4(acc_b[4 * m], acc_b[4 * m + 1], acc_b[4 * m + 2], acc_b[4 * m + 3]);
        });
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
        if ((tid & 31) == 0) p.sq_partials[slab_index * (T / 32) + (tid >> 5)] = sq;
    } else {
        // ------------------------------------------------------------------ Y role
        float s1r[PREG ? E : 1], s2r[PREG == 2 ? E : 1], gr[PREG ? E : 1];
        if constexpr (PREG > 0) {
            load_first_regs(p.s1, s1r);
            if constexpr (PREG == 2) load_first_regs(p.s2, s2r);
            load_g_regs(gr);
        }
        float acc_g[E], acc_2[E];
#pragma unroll
        for (int i = 0; i < E; ++i) acc_g[i] = acc_2[i] = 0.f;
#pragma unroll 1
        for (int it = 0; it < p.iters_per_group; ++it) {
            const int64_t e0 = tile_of(it, pair);
            if (e0 >= p.sample_elems) break;
            const int64_t left = p.sample_elems - e0;
            const int st = it % NS;
            const float* stage_x = pair_smem + size_t(st) * 2 * TILE;
            const float* stage_r = stage_x + TILE;
            const float* stash = stash0 + size_t(st) * TILE;
            mbar_wait(&ready_bar[pair][st], (it / NS) & 1);  // r, t2 (and, transitively, the TMA data) are visible
            float b[E];
            for_each_vec<N, C, V_FIRST>(off_f, cmask, [&](auto m_, uint32_t off, uint32_t coord) {
                constexpr int m = decltype(m_)::value;
                const float4 q = *reinterpret_cast<const float4*>(stage_r + off);
                mul4(b + 4 * m, q, first_param(s1r, p.s1, m, coord, PREG > 0));
            });
            to_mid(b);  // b = dt3
#pragma unroll
            for (int j = 0; j < E / 4; ++j) {  // dg += dt3 * t2
                const float4 t2 = *reinterpret_cast<const float4*>(stash + st_base + ((j ^ st_swz) << 2));
                fma4(acc_g + 4 * j, t2, b + 4 * j);
            }
            apply_g(b, gr);
            from_mid(b);  // b = dt1 (FIRST layout)
            const bool want_dx = p.dx != nullptr;
            IO* __restrict__ dxs = reinterpret_cast<IO*>(p.dx) + int64_t(s) * p.sample_elems + e0;
            for_each_vec<N, C, V_FIRST>(off_f, cmask, [&](auto m_, uint32_t off, uint32_t coord) {
                constexpr int m = decltype(m_)::value;
                const float4 q = Io<IO>::lds4(reinterpret_cast<const IO*>(stage_x) + off);
                const float4 w = first_param(s2r, p.s2, m, coord, PREG == 2);
                fma4(acc_2 + 4 * m, q, b + 4 * m);
                const float4 o = make_float4(q.x > relu_thr ? b[4 * m] * w.x : 0.f, q.y > relu_thr ? b[4 * m + 1] * w.y : 0.f,
                                             q.z > relu_thr ? b[4 * m + 2] * w.z : 0.f, q.w > relu_thr ? b[4 * m + 3] * w.w : 0.f);
                if (want_dx && (left >= TILE || off < left)) Io<IO>::st4(dxs + off, o);
            });
            mbar_arrive(&empty_bar[pair][st]);
        }
        // dg (middle layout) and ds2 (FIRST layout) partial sums -> workspace
        if constexpr (ROUNDS == 3) {
            for_each_vec<N, C, V_LAST>(off_l, cmask, [&](auto m_, uint32_t off, uint32_t) {
                constexpr int m = decltype(m_)::value;
                *reinterpret_cast<float4*>(slab + off) = make_float4(acc_g[4 * m], acc_g[4 * m + 1], acc_g[4 * m + 2], acc_g[4 * m + 3]);
            });
        } else {
            static_for<0, E>([&](auto r_) {
                constexpr int r = decltype(r_)::value;
                constexpr uint32_t rl = view_reg_logical(view_mid(N, C), r);
                slab[mid_logical | rl] = acc_g[r];
            });
        }
        for_each_vec<N, C, V_FIRST>(off_f, cmask, [&](auto m_, uint32_t off, uint32_t) {
            constexpr int m = decltype(m_)::value;
            *reinterpret_cast<float4*>(slab + 2 * TILE + off) = make_float4(acc_2[4 * m], acc_2[4 * m + 1], acc_2[4 * m + 2], acc_2[4 * m + 3]);
        });
    }
}

template <int N, int C, int KT, int PAIRS, int NS, bool SINGLE, int PREG, int ROUNDS>
static int launch_loss_cfg(const LayerLossCall& c, int k, cudaStream_t stream)
{
    static unsigned char smem_ok[4][64] = {};
    constexpr int T = 1 << (N - C);
    constexpr int threads = 2 * T * PAIRS;
    constexpr size_t tile = size_t(1) << N;
    constexpr size_t smem = sizeof(float) * ((2 * NS + NS) * tile + (SINGLE ? 2 : 4) * size_t(scratch_words(N, C))) * PAIRS;
    static_assert(smem <= 227 * 1024, "loss kernel shared memory");
    const int64_t D = int64_t(1) << k;
    const int64_t tiles_per_sample = (c.B * D + int64_t(tile) - 1) / int64_t(tile);
    const Plan plan = make_plan_waves(c.S, tiles_per_sample, PAIRS, 148, 8, 8);
    const int64_t slabs = int64_t(c.S) * plan.ctas_per_sample * PAIRS;
    const size_t need = sizeof(float) * size_t(slabs) * 4 * tile;
    if (c.need_ws) {
        *c.need_ws = need;
        *c.need_sq = slabs * (T / 32);
        return WHVI_OK;
    }
    if (c.ws == nullptr || c.ws_bytes < need)
        return fail(WHVI_E_WORKSPACE, "layer_loss: workspace of %zu bytes needed, %zu given", need, c.ws_bytes);
    const int64_t ctas = int64_t(plan.ctas_per_sample) * c.S;
    if (ctas > 0x7fffffffLL) return fail(WHVI_E_SHAPE, "layer_loss: grid too large");
    LossArgs a{c.x, c.xs, c.g, c.s1, c.s2, c.bias, c.target, c.dx, c.ws, c.sq_partials, c.B * D, static_cast<int>(c.S),
               plan.ctas_per_sample, plan.iters_per_group, k, c.relu_in};
    auto go = [&](auto kernel, int slot) -> int {
        if (int rc = ensure_smem(kernel, smem, smem_ok[slot])) return rc;
        kernel<<<static_cast<unsigned>(ctas), threads, smem, stream>>>(a);
        return check_launch("layer_loss_kernel");
    };
    const int rc = c.bf16 ? (c.bias ? go(layer_loss_kernel<N, C, KT, PAIRS, NS, SINGLE, PREG, ROUNDS, true, __nv_bfloat16>, 2)
                                    : go(layer_loss_kernel<N, C, KT, PAIRS, NS, SINGLE, PREG, ROUNDS, false, __nv_bfloat16>, 3))
                 : c.bias ? go(layer_loss_kernel<N, C, KT, PAIRS, NS, SINGLE, PREG, ROUNDS, true>, 0)
                          : go(layer_loss_kernel<N, C, KT, PAIRS, NS, SINGLE, PREG, ROUNDS, false>, 1);
    if (rc) return rc;
    return launch_bwd_reduce(c.ws, c.dg, c.ds1, c.ds2, c.bias ? c.dbias : nullptr, c.S, plan.ctas_per_sample * PAIRS, int64_t(tile), D, stream);
}

int launch_layer_loss(const LayerLossCall& c, int64_t D, cudaStream_t stream)
{
    const int k = ilog2(D);
#ifndef WHVI_LOSS_LEGACY   // -DWHVI_LOSS_LEGACY=1: round 1's three-view register-only kernel at D = 2048, 4096 (A/B builds)
    if ((k == 11 || k == 12) && c.need_ws) {
        // size query: the caller does not say whether there will be a bias, and the two kernels split the work
        // differently -> report the larger of each (unused sq_partials entries must be zero: see whvi_b200.h)
        size_t ws_a = 0, ws_b = 0;
        int64_t sq_a = 0, sq_b = 0;
        LayerLossCall q = c;
        q.need_ws = &ws_a, q.need_sq = &sq_a;
        if (int rc = launch_layer_loss_tm(q, D, stream)) return rc;
        q.need_ws = &ws_b, q.need_sq = &sq_b;
        const int rc = k == 11 ? launch_loss_cfg<11, 5, 11, 2, 3, false, 1, 3>(q, k, stream)
                               : launch_loss_cfg<12, 5, 12, 1, 3, false, 1, 3>(q, k, stream);
        if (rc) return rc;
        *c.need_ws = ws_a > ws_b ? ws_a : ws_b;
        *c.need_sq = sq_a > sq_b ? sq_a : sq_b;
        return WHVI_OK;
    }
    if ((k == 11 || k == 12) && c.bias == nullptr) return launch_layer_loss_tm(c, D, stream);
#endif
    if (k >= 7 && k <= 9) return launch_loss_cfg<10, 5, k_family(7, 9), 4, 3, false, 1, 2>(c, k, stream);
    if (k == 10) return launch_loss_cfg<10, 5, 10, 4, 3, false, 1, 2>(c, k, stream);
    if (k == 11) return launch_loss_cfg<11, 5, 11, 2, 3, false, 1, 3>(c, k, stream);
    if (k == 12) return launch_loss_cfg<12, 5, 12, 1, 3, false, 1, 3>(c, k, stream);
    return fail(WHVI_E_SHAPE, "layer_loss: D = %lld unsupported (128 <= D <= 4096)", (long long)D);
}

}  // namespace whvi
