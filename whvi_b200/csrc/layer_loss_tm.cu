// Fused LAST layer (forward + Gaussian-MNLL residual + backward, see layer_loss.cu for the math), TMEM edition for
// D = 2048, 4096 without a bias (round 2).
//
// Same two pipelined roles as layer_loss.cu -- X: t2 = H(s2 x) -> t4 = H(g t2) -> r = s1 t4 - target, sum r^2,
// ds1 += r t4;  Y, one tile behind: dt3 = H(s1 r) -> dg += dt3 t2 -> dt1 = H(g dt3) -> ds2 += dt1 x, dx = s2 dt1 --
// but with two views and 64 floats per thread (ONE transposition per transform instead of two: the round-1 kernel
// sat at 33% of the HBM roofline on the L1/shared-memory data pipe) and with everything that is private to a
// thread, or shared only by the X and Y threads of the same lane, in TENSOR MEMORY (tmem.cuh):
//   [0,E) g | [E,2E) s1 | [2E,3E) s2 | [3E,4E) ds1 (X) | [4E,5E) dg (Y) | [5E,6E) ds2 (Y) | [6E,8E) t2, two tiles deep
// so a thread's registers hold its 64-float stream and little else, t2 never touches shared memory, and two tile
// pairs (2 x 2 roles x 2 warps) fit on an SM: 3 x-tile slots + 2 target/r slots + one in-place transposition buffer
// per role = 112 KB per pair.  x and target tiles have separate rings because their lifetimes differ (x: X's start
// to Y's end, two tiles; target -> r: X's end to Y's start); the producer (thread 0 of X) refills an x slot at the
// END of its iteration, when Y has just released it, and a target slot in the MIDDLE.  One instruction stream per
// role section, shared transform code (the instruction cache holds ~32 KB; see layer_bwd.cu).
// This translation unit uses the XOR-swizzled transposition layout: the padded one needs 1 KB more than the 227 KB
// an SM has.
#include "layer_common.cuh"
#include "tmem.cuh"

namespace whvi {

// IO: the type of x and dx in HBM (see layer_loss_kernel): bf16 x tiles fill the first half of their fp32-sized slots.
template <int N, int C, int KT, class IO = float>
__global__ void __launch_bounds__(256, 1) layer_loss_tm_kernel(const LossArgs p)
{
    constexpr int T = 1 << (N - C);
    constexpr int E = 1 << C;
    constexpr int PAIRS = 128 / T;
    constexpr int NX = 3, NT = 2;
    constexpr int64_t TILE = int64_t(1) << N;
    constexpr int SW = int(scratch_words(N, C));
    constexpr int PAIR_FLOATS = (NX + NT) * int(TILE) + 2 * SW;
    static_assert(E == 64 && PAIRS * T == 128, "layer_loss_tm_kernel: 64 floats per thread, 4 warps per role");
    static_assert(rounds_needed(N, C, N) <= 2, "two views must cover every tile bit");
    constexpr uint32_t COL_G = 0, COL_S1 = E, COL_S2 = 2 * E, COL_A1 = 3 * E, COL_AG = 4 * E, COL_A2 = 5 * E, COL_T2 = 6 * E;
    extern __shared__ float4 smem4[];
    __shared__ uint64_t x_full[PAIRS][NX], x_empty[PAIRS][NX], t_full[PAIRS][NT], t_empty[PAIRS][NT], r_ready[PAIRS][NT],
        t2_free[PAIRS][2], reads_done[PAIRS][2];
    __shared__ uint32_t tmem_base_smem;
    float* smem = reinterpret_cast<float*>(smem4);
    const int k = KT >= 0 ? KT : p.k;
    const uint32_t cmask = (1u << k) - 1u;
    const int s = blockIdx.x % p.n_samples;  // sample-minor CTA order: the target tile is reused out of L2
    const int cta_in_sample = blockIdx.x / p.n_samples;
    const IO* __restrict__ xbase = reinterpret_cast<const IO*>(p.x) + int64_t(s) * p.x_sample_stride;

    if (threadIdx.x == 0) {
        for (int q = 0; q < PAIRS; ++q) {
            for (int i = 0; i < NX; ++i) mbar_init(&x_full[q][i], 1), mbar_init(&x_empty[q][i], T);
            for (int i = 0; i < NT; ++i) mbar_init(&t_full[q][i], 1), mbar_init(&t_empty[q][i], T), mbar_init(&r_ready[q][i], T);
            for (int i = 0; i < 2; ++i) mbar_init(&t2_free[q][i], T), mbar_init(&reads_done[q][i], T);
        }
        mbar_fence_init();
    }
    if (threadIdx.x < 32) tm_alloc(&tmem_base_smem, 512);
    tm_fence_before();
    __syncthreads();
    tm_fence_after();
    const uint32_t tm = tm_lane_base(tmem_base_smem);

    const int role = threadIdx.x / 128;               // 0 = X (warps 0..3), 1 = Y (warps 4..7): same TMEM lane per tid
    const int pair = (threadIdx.x % 128) / T;
    const uint32_t tid = threadIdx.x % T;
    float* pair_smem = smem + size_t(pair) * PAIR_FLOATS;
    float* xslots = pair_smem;                        // NX tiles
    float* tslots = pair_smem + NX * TILE;            // NT tiles: target on arrival, r after X's end section
    float* scratch = pair_smem + (NX + NT) * TILE + role * SW;
    const int bar_role = 1 + 2 * pair + role;
    const float* __restrict__ gs = p.g + (int64_t(s) << k);
    const float relu_thr = p.relu_in ? 0.f : -INFINITY;

    auto tile_of = [&](int it) -> int64_t { return ((int64_t(cta_in_sample) * p.iters_per_group + it) * PAIRS + pair) * TILE; };
    auto tile_bytes = [&](int it) -> uint32_t {   // 0: no such tile
        if (it >= p.iters_per_group) return 0;
        const int64_t e0 = tile_of(it);
        if (e0 >= p.sample_elems) return 0;
        const int64_t left = p.sample_elems - e0;
        return static_cast<uint32_t>((left < TILE ? left : TILE) * sizeof(float));
    };
    auto issue_x = [&](int it) {      // x tile `it` -> slot it % NX (waits for Y's release of tile it - NX)
        const uint32_t bytes = tile_bytes(it) / (sizeof(float) / sizeof(IO));
        if (!bytes) return;
        const int sl = it % NX;
        if (it >= NX) mbar_wait(&x_empty[pair][sl], ((it / NX) & 1) ^ 1);
        mbar_arrive_expect_tx(&x_full[pair][sl], bytes);
        bulk_g2s(xslots + size_t(sl) * TILE, xbase + tile_of(it), bytes, &x_full[pair][sl]);
    };
    auto issue_t = [&](int it) {      // target tile `it` -> slot it % NT (waits for Y's release of tile it - NT)
        const uint32_t bytes = tile_bytes(it);
        if (!bytes) return;
        const int sl = it % NT;
        if (it >= NT) mbar_wait(&t_empty[pair][sl], ((it / NT) & 1) ^ 1);
        mbar_arrive_expect_tx(&t_full[pair][sl], bytes);
        bulk_g2s(tslots + size_t(sl) * TILE, p.target + tile_of(it), bytes, &t_full[pair][sl]);
    };

    const uint32_t off_f = tile_thread_offset<N, C, V_FIRST>(tid);
    const uint32_t wb_fm = transpose_writer_base<N, C, V_FIRST, V_MID>(tid);
    const uint32_t wb_mf = transpose_writer_base<N, C, V_MID, V_FIRST>(tid);
    const uint32_t mid_logical = view_tid_logical(view_mid(N, C), tid);
    const int64_t slab_index = (int64_t(s) * p.ctas_per_sample + cta_in_sample) * PAIRS + pair;
    float* __restrict__ slab = p.ws + slab_index * 4 * TILE;

    // ---- TMEM initialisation: X writes g and s1 and zeroes ds1; Y writes s2 and zeroes dg, ds2
    {
        float z[32], w[E];
#pragma unroll
        for (int i = 0; i < 32; ++i) z[i] = 0.f;
        if (role == 0) {
            tm_st32(z, tm + COL_A1), tm_st32(z, tm + COL_A1 + 32);
            static_for<0, E>([&](auto r_) {
                constexpr int r = decltype(r_)::value;
                constexpr uint32_t rl = view_reg_logical(view_mid(N, C), r);
                w[r] = __ldg(gs + ((mid_logical | rl) & cmask));
            });
            tm_st32(w, tm + COL_G), tm_st32(w + 32, tm + COL_G + 32);
            tm_wait_st();
        } else {
            tm_st32(z, tm + COL_AG), tm_st32(z, tm + COL_AG + 32), tm_st32(z, tm + COL_A2), tm_st32(z, tm + COL_A2 + 32);
        }
        const float* __restrict__ pv = role ? p.s2 : p.s1;
        for_each_vec<N, C, V_FIRST>(off_f, cmask, [&](auto m_, uint32_t, uint32_t coord) {
            constexpr int m = decltype(m_)::value;
            const float4 q = ldg4(pv + coord);
            w[4 * m] = q.x, w[4 * m + 1] = q.y, w[4 * m + 2] = q.z, w[4 * m + 3] = q.w;
        });
        tm_st32(w, tm + (role ? COL_S2 : COL_S1)), tm_st32(w + 32, tm + (role ? COL_S2 : COL_S1) + 32);
        tm_wait_st();
        tm_fence_before();
        __syncthreads();
        tm_fence_after();
    }

    int it_now = 0;
    // stream (FIRST layout) -> middle layout and back: shared by both roles
    auto to_mid = [&](float (&v)[E]) {
        bfly_round<N, C, KT, SEQ2_IN, 0>(v, k);
        if (it_now > 0) mbar_wait(&reads_done[pair][role], (it_now - 1) & 1);   // the scratch has been read out (see layer_bwd.cu)
        transpose_write<N, C, V_FIRST, V_MID>(v, scratch, wb_fm);
        role_sync<T>(bar_role);
        transpose_read<C>(v, scratch, tid);
        bfly_round<N, C, KT, SEQ2_IN, 1>(v, k);
    };
    auto from_mid = [&](float (&v)[E]) {
        bfly_round<N, C, KT, SEQ2_OUT, 0>(v, k);
        role_sync<T>(bar_role);   // the first transposition has been read out by the whole role
        transpose_write<N, C, V_MID, V_FIRST>(v, scratch, wb_mf);
        role_sync<T>(bar_role);
        transpose_read<C>(v, scratch, tid);
        mbar_arrive(&reads_done[pair][role]);
        bfly_round<N, C, KT, SEQ2_OUT, 1>(v, k);
    };
    auto apply_g = [&](float (&v)[E]) {
#pragma unroll
        for (int c = 0; c < E; c += 32) {
            float gq[32];
            tm_ld32(gq, tm + COL_G + c);
            tm_wait_ld();
#pragma unroll
            for (int m = 0; m < 8; ++m) scale4(v + c + 4 * m, make_float4(gq[4 * m], gq[4 * m + 1], gq[4 * m + 2], gq[4 * m + 3]));
        }
    };
    // v = param (TMEM columns `col`, FIRST order) * tile (shared memory, FIRST layout)
    auto load_scaled = [&](float (&v)[E], const float* tile, uint32_t col) {
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            float w[32];
            tm_ld32(w, tm + col + 32 * c);
            float4 q[8];
            static_for<0, 8>([&](auto j_) {
                constexpr int j = decltype(j_)::value;
                q[j] = *reinterpret_cast<const float4*>(tile + off_f + tile_reg_offset<N, C, V_FIRST>(8 * c + j));
            });
            tm_wait_ld();
#pragma unroll
            for (int j = 0; j < 8; ++j) mul4(v + 32 * c + 4 * j, q[j], make_float4(w[4 * j], w[4 * j + 1], w[4 * j + 2], w[4 * j + 3]));
        }
    };
    // the same for the X role's x tile when x is bf16 (IO != float): widened on the read
    auto load_scaled_io = [&](float (&v)[E], const IO* tile, uint32_t col) {
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            float w[32];
            tm_ld32(w, tm + col + 32 * c);
            float4 q[8];
            static_for<0, 8>([&](auto j_) {
                constexpr int j = decltype(j_)::value;
                q[j] = Io<IO>::lds4(tile + off_f + tile_reg_offset<N, C, V_FIRST>(8 * c + j));
            });
            tm_wait_ld();
#pragma unroll
            for (int j = 0; j < 8; ++j) mul4(v + 32 * c + 4 * j, q[j], make_float4(w[4 * j], w[4 * j + 1], w[4 * j + 2], w[4 * j + 3]));
        }
    };

    // ONE loop for both roles: the two transforms and the g multiply are the same instructions on different data, and a
    // private copy per role does not fit the instruction cache next to the other role's (39% of the warp samples of the
    // first version were "no instruction" stalls, profiles/r02_bwd_notes.md).  Role-specific: what is waited for, the
    // middle section (X parks t2 / Y accumulates dg) and the end section (X: residual, Y: dx).
    float sq = 0.f;
    if (role == 0 && tid == 0) {
        issue_x(0), issue_x(1);
        issue_t(0);
    }
    const uint32_t col_in = role ? COL_S1 : COL_S2;
#pragma unroll 1
    for (int it = 0; it < p.iters_per_group; ++it) {
        const int64_t e0 = tile_of(it);
        if (e0 >= p.sample_elems) break;
        const int64_t left = p.sample_elems - e0;
        float* xt = xslots + size_t(it % NX) * TILE;
        float* tt = tslots + size_t(it % NT) * TILE;   // target, then r
        if (role == 0) {
            mbar_wait(&x_full[pair][it % NX], (it / NX) & 1);
            if (left < TILE) {  // partial tile: zero this thread's float4s beyond the valid part of x
                static_for<0, E / 4>([&](auto m_) {
                    constexpr int m = decltype(m_)::value;
                    const uint32_t off = off_f + tile_reg_offset<N, C, V_FIRST>(m);
                    if (off >= left) Io<IO>::sts_zero4(reinterpret_cast<IO*>(xt) + off);
                });
            }
        } else {
            mbar_wait(&r_ready[pair][it % NT], (it / NT) & 1);   // r, t2 (and, transitively, the x tile) are visible
            tm_fence_after();
        }
        float v[E];
        if constexpr (std::is_same_v<IO, float>) load_scaled(v, role ? tt : xt, col_in);   // X: s2 * x, Y: s1 * r
        else if (role) load_scaled(v, tt, col_in);
        else load_scaled_io(v, reinterpret_cast<const IO*>(xt), col_in);
        if (role) mbar_arrive(&t_empty[pair][it % NT]);   // r has been read: the slot may take the next target tile
        it_now = it;
        to_mid(v);  // X: t2, Y: dt3
        if (role == 0) {
            if (tid == 0) issue_t(it + 1);   // its slot was released at Y's start of tile it - 1
            if (it >= 2) mbar_wait(&t2_free[pair][it & 1], ((it - 2) >> 1) & 1);   // Y has read t2 of tile it - 2
            tm_fence_after();
            tm_st32(v, tm + COL_T2 + E * (it & 1)), tm_st32(v + 32, tm + COL_T2 + E * (it & 1) + 32);
        } else {
#pragma unroll
            for (int c = 0; c < 2; ++c) {   // dg += dt3 * t2
                float t2[32], ag[32];
                tm_ld32(t2, tm + COL_T2 + E * (it & 1) + 32 * c);
                tm_ld32(ag, tm + COL_AG + 32 * c);
                tm_wait_ld();
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    fma4(ag + 4 * j, make_float4(t2[4 * j], t2[4 * j + 1], t2[4 * j + 2], t2[4 * j + 3]), v + 32 * c + 4 * j);
                tm_st32(ag, tm + COL_AG + 32 * c);
            }
            tm_fence_before();
            mbar_arrive(&t2_free[pair][it & 1]);
        }
        apply_g(v);
        from_mid(v);  // X: t4, Y: dt1 (FIRST layout)
        if (role == 0) {
            mbar_wait(&t_full[pair][it % NT], (it / NT) & 1);
#pragma unroll
            for (int c = 0; c < 2; ++c) {   // y_hat = s1 t4, r = y_hat - target, sum r^2, ds1 += r t4, r -> Y
                float w[32], a1[32];
                tm_ld32(w, tm + COL_S1 + 32 * c);
                tm_ld32(a1, tm + COL_A1 + 32 * c);
                float4 tg[8];
                static_for<0, 8>([&](auto j_) {
                    constexpr int j = decltype(j_)::value;
                    tg[j] = *reinterpret_cast<const float4*>(tt + off_f + tile_reg_offset<N, C, V_FIRST>(8 * c + j));
                });
                tm_wait_ld();
                static_for<0, 8>([&](auto j_) {
                    constexpr int j = decltype(j_)::value;
                    const uint32_t off = off_f + tile_reg_offset<N, C, V_FIRST>(8 * c + j);
                    const float* t4 = v + 32 * c + 4 * j;
                    const bool valid = left >= TILE || off < left;
                    const float4 r = valid ? make_float4(t4[0] * w[4 * j] - tg[j].x, t4[1] * w[4 * j + 1] - tg[j].y,
                                                         t4[2] * w[4 * j + 2] - tg[j].z, t4[3] * w[4 * j + 3] - tg[j].w)
                                           : make_float4(0.f, 0.f, 0.f, 0.f);
                    sq = fmaf(r.x, r.x, fmaf(r.y, r.y, fmaf(r.z, r.z, fmaf(r.w, r.w, sq))));
                    fma4(a1 + 4 * j, r, t4);
                    *reinterpret_cast<float4*>(tt + off) = r;
                });
                tm_st32(a1, tm + COL_A1 + 32 * c);
            }
            tm_wait_st();          // t2 and ds1 are in tensor memory ...
            tm_fence_before();
            mbar_arrive(&r_ready[pair][it % NT]);   // ... and r in shared memory: released to the Y role
            if (tid == 0) issue_x(it + 2);   // refill the x slot Y released at the end of tile it - 1
        } else {
            mbar_wait(&x_full[pair][it % NX], (it / NX) & 1);   // completed long ago; orders this thread after the bulk copy
            const bool want_dx = p.dx != nullptr;
            IO* __restrict__ dxs = reinterpret_cast<IO*>(p.dx) + int64_t(s) * p.sample_elems + e0;
#pragma unroll
            for (int c = 0; c < 2; ++c) {   // ds2 += dt1 * x, dx = s2 * dt1 (masked)
                float w[32], a2[32];
                tm_ld32(w, tm + COL_S2 + 32 * c);
                tm_ld32(a2, tm + COL_A2 + 32 * c);
                float4 q[8];
                static_for<0, 8>([&](auto j_) {
                    constexpr int j = decltype(j_)::value;
                    q[j] = Io<IO>::lds4(reinterpret_cast<const IO*>(xt) + off_f + tile_reg_offset<N, C, V_FIRST>(8 * c + j));
                });
                tm_wait_ld();
                static_for<0, 8>([&](auto j_) {
                    constexpr int j = decltype(j_)::value;
                    const uint32_t off = off_f + tile_reg_offset<N, C, V_FIRST>(8 * c + j);
                    const float* bb = v + 32 * c + 4 * j;
                    fma4(a2 + 4 * j, q[j], bb);
                    const float4 o = make_float4(q[j].x > relu_thr ? bb[0] * w[4 * j] : 0.f, q[j].y > relu_thr ? bb[1] * w[4 * j + 1] : 0.f,
                                                 q[j].z > relu_thr ? bb[2] * w[4 * j + 2] : 0.f, q[j].w > relu_thr ? bb[3] * w[4 * j + 3] : 0.f);
                    if (want_dx && (left >= TILE || off < left)) Io<IO>::st4(dxs + off, o);
                });
                tm_st32(a2, tm + COL_A2 + 32 * c);
            }
            mbar_arrive(&x_empty[pair][it % NX]);
            tm_wait_st();
        }
    }
    if (role == 0) {
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            float a1[32];
            tm_ld32(a1, tm + COL_A1 + 32 * c);
            tm_wait_ld();
            static_for<0, 8>([&](auto j_) {
                constexpr int j = decltype(j_)::value;
                const uint32_t off = off_f + tile_reg_offset<N, C, V_FIRST>(8 * c + j);
                *reinterpret_cast<float4*>(slab + TILE + off) = make_float4(a1[4 * j], a1[4 * j + 1], a1[4 * j + 2], a1[4 * j + 3]);
            });
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
        if ((tid & 31) == 0) p.sq_partials[slab_index * (T / 32) + (tid >> 5)] = sq;
    } else {
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            float a[32];
            tm_ld32(a, tm + COL_AG + 32 * c);
            tm_wait_ld();
            static_for<0, 32>([&](auto r_) {   // dg: middle-layout register order -> tile coordinates
                constexpr int r = decltype(r_)::value;
                slab[mid_logical | view_reg_logical(view_mid(N, C), 32 * c + r)] = a[r];
            });
            tm_ld32(a, tm + COL_A2 + 32 * c);
            tm_wait_ld();
            static_for<0, 8>([&](auto j_) {
                constexpr int j = decltype(j_)::value;
                const uint32_t off = off_f + tile_reg_offset<N, C, V_FIRST>(8 * c + j);
                *reinterpret_cast<float4*>(slab + 2 * TILE + off) = make_float4(a[4 * j], a[4 * j + 1], a[4 * j + 2], a[4 * j + 3]);
            });
        }
    }
    tm_fence_before();
    __syncthreads();
    if (threadIdx.x < 32) tm_dealloc(tmem_base_smem, 512);
}

template <int N, int C, int KT>
static int launch_loss_tm_cfg(const LayerLossCall& c, int k, cudaStream_t stream)
{
    static unsigned char smem_ok[2][64] = {};
    constexpr int T = 1 << (N - C);
    constexpr int PAIRS = 128 / T;
    constexpr size_t tile = size_t(1) << N;
    constexpr size_t smem = sizeof(float) * PAIRS * (5 * tile + 2 * size_t(scratch_words(N, C)));
    static_assert(smem + 1024 <= 227 * 1024, "TMEM loss kernel shared memory");
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
        kernel<<<static_cast<unsigned>(ctas), 256, smem, stream>>>(a);
        return check_launch("layer_loss_tm_kernel");
    };
    if (int rc = c.bf16 ? go(layer_loss_tm_kernel<N, C, KT, __nv_bfloat16>, 1) : go(layer_loss_tm_kernel<N, C, KT>, 0)) return rc;
    return launch_bwd_reduce(c.ws, c.dg, c.ds1, c.ds2, nullptr, c.S, plan.ctas_per_sample * PAIRS, int64_t(tile), D, stream);
}

int launch_layer_loss_tm(const LayerLossCall& c, int64_t D, cudaStream_t stream)
{
    const int k = ilog2(D);
    if (k == 11) return launch_loss_tm_cfg<12, 6, 11>(c, k, stream);
    if (k == 12) return launch_loss_tm_cfg<12, 6, 12>(c, k, stream);
    return fail(WHVI_E_SHAPE, "layer_loss(tm): D = %lld unsupported", (long long)D);
}

}  // namespace whvi
