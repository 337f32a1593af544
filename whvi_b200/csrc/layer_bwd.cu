// Kernel (3): the fused WHVILinear backward (see layer_fwd.cu for the math and layout notes).
// The transposition buffers of THIS translation unit use the padded (XOR-free) layout: the backward gains ~4% at
// D = 1024...8192 over the swizzled one with bit-identical outputs, the two-view forward does not
// (profiles/r01_bwd_notes.md item 14, profiles/r02_ab_padbwd.txt).
#define WHVI_PADDED 1
#include "layer_common.cuh"
#include "tmem.cuh"

namespace whvi {

// ------------------------------------------------------------------------------ backward
// Shared memory of layer_bwd_tma_kernel: per tile pair, 2 stages of `spt` tiles, a half-stash pair (one tile) and two
// transposition buffers per role.  Does the MNLL target tile ride in the TMA stage (RESID kernels)?  One definition for
// the kernel's shared-memory carve-up and the launcher's size computation.
// sw = words of one transposition buffer (scratch_words(n, c))
constexpr size_t bwd_smem_bytes(int n, int pairs, int spt, size_t sw)
{
    return sizeof(float) * ((size_t(spt) * 2 + 1) * (size_t(1) << n) + 4 * sw) * pairs;
}
constexpr bool bwd_stage_target(int n, int pairs, size_t sw) { return bwd_smem_bytes(n, pairs, 3, sw) <= size_t(200) * 1024; }

struct BwdArgs {
    const float* x;
    int64_t x_sample_stride;
    const float* dy;       // (S,B,D) upstream gradient, or -- RESID -- the layer's saved output
    const float* g;
    const float* s1;
    const float* s2;
    float* dx;             // NULL: skip
    float* ws;
    int64_t sample_elems;
    int n_samples;          // S
    int ctas_per_sample;
    int iters_per_group;
    int k;                 // log2(D)
    int relu_in;           // x is the output of a fused ReLU: dx *= (x > 0)
    const float* target;   // RESID: (B,D); dy := coef[0] * (dy_buffer - target)  (fused Gaussian-MNLL gradient)
    const float* coef;     // RESID: device scalar
    const float* dy_scale; // optional device scalar: the upstream gradient is dy_scale[0] * dy (deferred
                           // scaling of a producer that computed its dx for a unit loss coefficient)
    int pad = 0;           // not read: keeps spg and pstride at the parameter offsets the kernels were timed with; without
                           // it ptxas allocates the registers of every backward instance differently (and
                           // layer_bwd_tm_kernel's RESID instances spill more)
    int spg = 0x7fffffff;  // grouped launch (LayerFwdCall): samples per parameter group
    int pstride = 0;       // floats between consecutive groups' s1 / s2 vectors
};

// Stream-role specialised, TMA-staged backward, D <= 1024.  Every tile is worked on by a PAIR of
// thread sets running concurrently:
//   X role:  t2 = H(s2*x) -> t4 = H(g*t2) -> ds1 += dy*t4 (+ dbias += dy)
//   Y role:  dt3 = H(s1*dy) -> dt1 = H(g*dt3) -> ds2 += dt1*x, dx = s2*dt1
//   both:    dg += dt3*t2, half of the coordinates each (exchanged through a half-stash)
// Each role keeps one stream (32 floats per thread) and its accumulators in registers.
// One CTA owns `iters_per_group * PAIRS` consecutive tiles of ONE sample; at the end every
// role writes its partial sums to the workspace and a second kernel reduces them in a fixed
// order (deterministic, no atomics).
// workspace layout: [S][ctas_per_sample][PAIRS][4][TILE] floats: 0 = dg, 1 = ds1, 2 = ds2, 3 = dbias
//
// One elected thread per pair streams the raw
// x and dy tiles into a ring of shared-memory stages with bulk async copies (mbarrier
// completion), NS tiles ahead of the compute roles.  Consequences:
//   * global-load latency is off the critical path (no registers hold loads in flight);
//   * each role reads BOTH raw tiles from shared memory (its own stream at the start, the
//     other stream for its end product), so x and dy cross HBM->SM exactly once (an earlier
//     register-staged variant re-read them through L2 and ~40% of those re-reads missed;
//     profiles/r01_bwd_notes.md);
//   * the dg accumulator is split between the roles (X: float4 slots 0..E/8-1, Y: the rest;
//     each sends the other the half-stream it needs through a shared half-stash), which
//     balances the register budgets of the two roles.
// One CTA per SM (shared memory is the limit), so the spare registers hold this thread's input-side
// scaling (X: s2, Y: s1) and g values across tiles.  A two-CTA/SM variant with shared-memory accumulators, a two-view
// 64-float variant and a single-barrier stash exchange were measured and dropped
// (profiles/r01_bwd_notes.md, items 5, 8, 10).
// Shared memory per pair: NS x (x tile + dy tile) + X scratch + Y scratch + stash (1 tile).
// IO: the activations' type in HBM (x, dy, dx; see layer_fwd_kernel).  bf16 tiles are staged in the first half of their
// fp32-sized slots (the plan, shared memory and partial-sum order are the fp32 instance's), widened on every read, and dx
// is rounded once at the store.  The workspace, the parameters and all arithmetic stay fp32; RESID is fp32 only.
// DX: the type dx is stored as (IO by default).  bf16 x and dy with an fp32 dx serve the grouped (Stacked) backward, whose
// per-block dx are summed in fp32 and rounded once by the caller.
template <int N, int C, int KT, bool WANT_DBIAS, bool RESID, class IO = float, class DX = IO>
__global__ void __launch_bounds__(256, 1) layer_bwd_tma_kernel(const BwdArgs p)
{
    static_assert(std::is_same_v<IO, float> || !RESID, "RESID (saved output + target) is fp32 only");
    constexpr int T = 1 << (N - C);
    constexpr int E = 1 << C;
    constexpr int H = E / 2;               // floats per thread per half-stream
    constexpr int PAIRS = 128 / T;
    constexpr int NS = 2;
    constexpr int64_t TILE = int64_t(1) << N;
    static_assert(PAIRS * T == 128, "layer_bwd_tma_kernel: 4 warps per role");
    // Two views: FIRST + MID cover every bit, and the middle of the layer (g multiply, dg products) is
    // the MID view -- half the transpositions of a three-view form, hence half of the dominant L1/shared wavefronts.
    static_assert(rounds_needed(N, C, N) <= 2, "2-view kernel needs FIRST+MID to cover all bits");
    constexpr int SW = int(scratch_words(N, C));  // one transposition buffer
    // RESID: the target tile rides in the stage too (third tile) when shared memory allows
    constexpr bool STAGE_TGT = RESID && bwd_stage_target(N, PAIRS, SW);
    constexpr int SPT = STAGE_TGT ? 3 : 2;   // tiles per stage
    constexpr int PAIR_FLOATS = (SPT * NS + 1) * int(TILE) + 4 * SW;
    extern __shared__ float4 smem4[];
    __shared__ uint64_t full_bar[PAIRS][NS], empty_bar[PAIRS][NS];
    float* smem = reinterpret_cast<float*>(smem4);
    const int k = KT >= 0 ? KT : p.k;
    const uint32_t cmask = (1u << k) - 1u;
    // sample-minor CTA order (see layer_fwd.cu): shared x / target tiles are reused out of L2
    const int s = blockIdx.x % p.n_samples;
    const int cta_in_sample = blockIdx.x / p.n_samples;
    const int grp = s / p.spg;   // parameter group (Stacked block); the group's virtual samples read the inputs of samples 0 .. spg-1
    const IO* __restrict__ xbase = reinterpret_cast<const IO*>(p.x) + int64_t(s - grp * p.spg) * p.x_sample_stride;
    const float* __restrict__ s1p = p.s1 + int64_t(grp) * p.pstride;
    const float* __restrict__ s2p = p.s2 + int64_t(grp) * p.pstride;
    const IO* __restrict__ dybase = reinterpret_cast<const IO*>(p.dy) + int64_t(s) * p.sample_elems;

    if (threadIdx.x == 0) {
        for (int q = 0; q < PAIRS; ++q)
            for (int st = 0; st < NS; ++st) {
                mbar_init(&full_bar[q][st], 1);
                mbar_init(&empty_bar[q][st], 2 * T);
            }
        mbar_fence_init();
    }
    __syncthreads();

    auto tile_of = [&](int it, int pr) -> int64_t {
        return ((int64_t(cta_in_sample) * p.iters_per_group + it) * PAIRS + pr) * TILE;
    };

    // In-band producer: thread 0 of each pair's X role issues the bulk copies for tile `it`
    // (both raw tiles, plus the target tile when staged) into stage it % NS.  It is called
    // one tile ahead; the wait on `empty` is for the other role to have finished tile it - NS,
    // which it does without depending on this thread (no deadlock), and this role would have
    // to wait for the other at the next pair barrier anyway.
    auto issue_tile = [&](int it, int pr) {
        if (it >= p.iters_per_group) return;
        const int64_t e0 = tile_of(it, pr);
        if (e0 >= p.sample_elems) return;
        const int st = it % NS;
        if (it >= NS) mbar_wait(&empty_bar[pr][st], ((it / NS) & 1) ^ 1);
        const int64_t left = p.sample_elems - e0;
        const uint32_t bytes = static_cast<uint32_t>((left < TILE ? left : TILE) * sizeof(IO));
        float* stage = smem + size_t(pr) * PAIR_FLOATS + size_t(st) * SPT * TILE;
        mbar_arrive_expect_tx(&full_bar[pr][st], SPT * bytes);
        bulk_g2s(stage, xbase + e0, bytes, &full_bar[pr][st]);
        bulk_g2s(stage + TILE, dybase + e0, bytes, &full_bar[pr][st]);
        if constexpr (STAGE_TGT) bulk_g2s(stage + 2 * TILE, p.target + e0, bytes, &full_bar[pr][st]);
    };

    const int role = threadIdx.x / (T * PAIRS);        // 0 = X, 1 = Y (warp-uniform)
    const int pair = (threadIdx.x % (T * PAIRS)) / T;
    const uint32_t tid = threadIdx.x % T;
    float* pair_smem = smem + size_t(pair) * PAIR_FLOATS;
    float* scratch = pair_smem + (SPT * NS) * TILE + (2 * role) * SW;  // this role's ping-pong transposition buffers
    float* scratch2 = scratch + SW;
    // half-stashes: X -> Y upper half of t2, Y -> X lower half of dt3
    float* stash_t2 = pair_smem + (SPT * NS) * TILE + 4 * SW;
    float* stash_d3 = stash_t2 + TILE / 2;
    const int bar_role = 1 + 3 * pair + role;
    const int bar_pair = 3 + 3 * pair;
    const float* __restrict__ gs = p.g + (int64_t(s) << k);
    float coef = 1.f;
    if constexpr (RESID) coef = __ldg(p.coef);
    const float dysc = p.dy_scale != nullptr ? __ldg(p.dy_scale) : 1.f;
    const float relu_thr = p.relu_in ? 0.f : -INFINITY;

    const uint32_t off_f = tile_thread_offset<N, C, V_FIRST>(tid);
    const uint32_t wb_fm = transpose_writer_base<N, C, V_FIRST, V_MID>(tid);
    const uint32_t wb_mf = transpose_writer_base<N, C, V_MID, V_FIRST>(tid);
    const uint32_t mid_logical = view_tid_logical(view_mid(N, C), tid);  // this thread's MID-view index bits
    // stream -> middle layout (t2 / dt3) and back (t4 / dt1)
    auto to_mid = [&](float (&v)[E]) {
        bfly_round<N, C, KT, SEQ2_IN, 0>(v, k);
        transpose_write<N, C, V_FIRST, V_MID>(v, scratch, wb_fm);
        role_sync<T>(bar_role);
        transpose_read<C>(v, scratch, tid);
        bfly_round<N, C, KT, SEQ2_IN, 1>(v, k);
    };
    auto from_mid = [&](float (&v)[E]) {
        bfly_round<N, C, KT, SEQ2_OUT, 0>(v, k);
        transpose_write<N, C, V_MID, V_FIRST>(v, scratch2, wb_mf);
        role_sync<T>(bar_role);
        transpose_read<C>(v, scratch2, tid);
        bfly_round<N, C, KT, SEQ2_OUT, 1>(v, k);
    };
    // g in the middle layout, once into registers
    auto load_g_regs = [&](float* gr) {
        static_for<0, E>([&](auto r_) {
            constexpr int r = decltype(r_)::value;
            constexpr uint32_t rl = view_reg_logical(view_mid(N, C), r);
            gr[r] = __ldg(gs + ((mid_logical | rl) & cmask));
        });
    };
    auto apply_g = [&](float (&v)[E], const float* gr) {
#pragma unroll
        for (int m = 0; m < E / 4; ++m) scale4(v + 4 * m, make_float4(gr[4 * m], gr[4 * m + 1], gr[4 * m + 2], gr[4 * m + 3]));
    };
    // this role's half of the dg partial sums -> workspace (registers [half*H, half*H + H))
    auto store_dg_half = [&](const float (&acc)[E / 2], int half_is_upper, float* dst) {
        static_for<0, E / 2>([&](auto r_) {
            constexpr int r = decltype(r_)::value;
            constexpr uint32_t rl_lo = view_reg_logical(view_mid(N, C), r);
            constexpr uint32_t rl_hi = view_reg_logical(view_mid(N, C), r + E / 2);
            dst[mid_logical | (half_is_upper ? rl_hi : rl_lo)] = acc[r];
        });
    };
    float* __restrict__ slab = p.ws + (((int64_t(s) * p.ctas_per_sample + cta_in_sample) * PAIRS + pair) * 4) * TILE;
    const uint32_t hs_base = tid << (C - 1);           // this thread's H floats in a half-stash
    const uint32_t hs_swz = swz_of_tid(C - 1, tid);

    // A partial tile (only at the tail of a sample) leaves stale data in the unfilled part of
    // the stage; instead of masking every read, each thread zero-fills its own float4s beyond
    // `left` in both raw tiles once per such tile (X and Y threads with the same tid own the
    // same offsets and both write zeros, which is benign).
    auto zero_tail = [&](float* stage_x, int64_t left) {
        if (left < TILE) {
            static_for<0, E / 4>([&](auto m_) {
                constexpr int m = decltype(m_)::value;
                const uint32_t off = off_f + tile_reg_offset<N, C, V_FIRST>(m);
                if (off >= left) {
                    Io<IO>::sts_zero4(reinterpret_cast<IO*>(stage_x) + off);
                    Io<IO>::sts_zero4(reinterpret_cast<IO*>(stage_x + TILE) + off);
                    if constexpr (STAGE_TGT) *reinterpret_cast<float4*>(stage_x + 2 * TILE + off) = make_float4(0.f, 0.f, 0.f, 0.f);
                }
            });
        }
    };
    auto raw4 = [&](const float* stage_tile, uint32_t off) -> float4 {
        return Io<IO>::lds4(reinterpret_cast<const IO*>(stage_tile) + off);
    };
    // RESID: dy = coef * (saved output - target); the target tile is read from global memory
    // (it is shared by all samples, so it stays L2-resident), zero beyond the valid part
    auto to_dy = [&](float4 q, const float* tgt, uint32_t off, int64_t left) -> float4 {
        if constexpr (RESID) {
            float4 tg = make_float4(0.f, 0.f, 0.f, 0.f);
            if constexpr (STAGE_TGT) {
                tg = *reinterpret_cast<const float4*>(tgt + off);  // tgt = the staged target tile
            } else if (left >= TILE || off < left) {
                tg = ldg4(tgt + off);
            }
            q = make_float4(coef * (q.x - tg.x), coef * (q.y - tg.y), coef * (q.z - tg.z), coef * (q.w - tg.w));
        } else {
            q = make_float4(dysc * q.x, dysc * q.y, dysc * q.z, dysc * q.w);
        }
        return q;
    };

    float acc_g[H];
#pragma unroll
    for (int i = 0; i < H; ++i) acc_g[i] = 0.f;

    if (role == 0) {
        // ------------------------------------------------------------------ X role
        // this thread's s2 and g values never change from tile to tile (its coordinates are
        // fixed), so they are loaded once; each per-tile parameter load otherwise costs as many
        // L1 wavefronts as a raw-tile read, and the L1/shared data pipe is what bounds this kernel
        float s2r[E], gr[E];
        for_each_vec<N, C, V_FIRST>(off_f, cmask, [&](auto m_, uint32_t, uint32_t coord) {
            constexpr int m = decltype(m_)::value;
            const float4 w = ldg4(s2p + coord);
            s2r[4 * m] = w.x, s2r[4 * m + 1] = w.y, s2r[4 * m + 2] = w.z, s2r[4 * m + 3] = w.w;
        });
        load_g_regs(gr);
        float acc_1[E];
        float acc_b[WANT_DBIAS ? E : 1];
#pragma unroll
        for (int i = 0; i < E; ++i) acc_1[i] = 0.f;
        if constexpr (WANT_DBIAS) {
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
            float* stage_x = pair_smem + size_t(st) * SPT * TILE;
            const float* stage_dy = stage_x + TILE;
            const float* tgt = STAGE_TGT ? stage_x + 2 * TILE : (RESID ? p.target + e0 : nullptr);
            if (tid == 0) issue_tile(it + NS - 1, pair);
            mbar_wait(&full_bar[pair][st], (it / NS) & 1);
            zero_tail(stage_x, left);
            float a[E];
            for_each_vec<N, C, V_FIRST>(off_f, cmask, [&](auto m_, uint32_t off, uint32_t) {
                constexpr int m = decltype(m_)::value;
                const float4 q = raw4(stage_x, off);
                mul4(a + 4 * m, q, make_float4(s2r[4 * m], s2r[4 * m + 1], s2r[4 * m + 2], s2r[4 * m + 3]));
            });
            to_mid(a);  // a = t2 (middle layout)
#pragma unroll
            for (int jj = 0; jj < H / 4; ++jj)   // publish the upper half of t2
                *reinterpret_cast<float4*>(stash_t2 + hs_base + ((jj ^ hs_swz) << 2)) =
                    make_float4(a[H + 4 * jj], a[H + 4 * jj + 1], a[H + 4 * jj + 2], a[H + 4 * jj + 3]);
            bar_wait<2 * T>(bar_pair);
#pragma unroll
            for (int jj = 0; jj < H / 4; ++jj) {  // dg (lower half) += dt3 * t2
                const float4 d = *reinterpret_cast<const float4*>(stash_d3 + hs_base + ((jj ^ hs_swz) << 2));
                fma4(acc_g + 4 * jj, d, a + 4 * jj);
            }
            bar_wait<2 * T>(bar_pair);  // both half-stashes consumed
            apply_g(a, gr);
            from_mid(a);  // a = t4 (FIRST layout)
            for_each_vec<N, C, V_FIRST>(off_f, cmask, [&](auto m_, uint32_t off, uint32_t) {
                constexpr int m = decltype(m_)::value;
                const float4 q = to_dy(raw4(stage_dy, off), tgt, off, left);
                fma4(acc_1 + 4 * m, q, a + 4 * m);
                if constexpr (WANT_DBIAS) {
                    acc_b[4 * m + 0] += q.x;
                    acc_b[4 * m + 1] += q.y;
                    acc_b[4 * m + 2] += q.z;
                    acc_b[4 * m + 3] += q.w;
                }
            });
            mbar_arrive(&empty_bar[pair][st]);
        }
        for_each_vec<N, C, V_FIRST>(off_f, cmask, [&](auto m_, uint32_t off, uint32_t) {
            constexpr int m = decltype(m_)::value;
            *reinterpret_cast<float4*>(slab + TILE + off) = make_float4(acc_1[4 * m], acc_1[4 * m + 1], acc_1[4 * m + 2], acc_1[4 * m + 3]);
            if constexpr (WANT_DBIAS)
                *reinterpret_cast<float4*>(slab + 3 * TILE + off) = make_float4(acc_b[4 * m], acc_b[4 * m + 1], acc_b[4 * m + 2], acc_b[4 * m + 3]);
        });
        store_dg_half(acc_g, 0, slab);
    } else {
        // ------------------------------------------------------------------ Y role
        float s1r[E], gr[E];   // s2 (for dx) is read per tile
        for_each_vec<N, C, V_FIRST>(off_f, cmask, [&](auto m_, uint32_t, uint32_t coord) {
            constexpr int m = decltype(m_)::value;
            const float4 w = ldg4(s1p + coord);
            s1r[4 * m] = w.x, s1r[4 * m + 1] = w.y, s1r[4 * m + 2] = w.z, s1r[4 * m + 3] = w.w;
        });
        load_g_regs(gr);
        float acc_2[E];
#pragma unroll
        for (int i = 0; i < E; ++i) acc_2[i] = 0.f;
#pragma unroll 1
        for (int it = 0; it < p.iters_per_group; ++it) {
            const int64_t e0 = tile_of(it, pair);
            if (e0 >= p.sample_elems) break;
            const int64_t left = p.sample_elems - e0;
            const int st = it % NS;
            float* stage_x = pair_smem + size_t(st) * SPT * TILE;
            const float* stage_dy = stage_x + TILE;
            const float* tgt = STAGE_TGT ? stage_x + 2 * TILE : (RESID ? p.target + e0 : nullptr);
            mbar_wait(&full_bar[pair][st], (it / NS) & 1);
            zero_tail(stage_x, left);
            float b[E];
            for_each_vec<N, C, V_FIRST>(off_f, cmask, [&](auto m_, uint32_t off, uint32_t) {
                constexpr int m = decltype(m_)::value;
                const float4 q = to_dy(raw4(stage_dy, off), tgt, off, left);
                mul4(b + 4 * m, q, make_float4(s1r[4 * m], s1r[4 * m + 1], s1r[4 * m + 2], s1r[4 * m + 3]));
            });
            to_mid(b);  // b = dt3 (middle layout)
#pragma unroll
            for (int jj = 0; jj < H / 4; ++jj)   // publish the lower half of dt3
                *reinterpret_cast<float4*>(stash_d3 + hs_base + ((jj ^ hs_swz) << 2)) =
                    make_float4(b[4 * jj], b[4 * jj + 1], b[4 * jj + 2], b[4 * jj + 3]);
            bar_wait<2 * T>(bar_pair);
#pragma unroll
            for (int jj = 0; jj < H / 4; ++jj) {  // dg (upper half) += dt3 * t2
                const float4 t2 = *reinterpret_cast<const float4*>(stash_t2 + hs_base + ((jj ^ hs_swz) << 2));
                fma4(acc_g + 4 * jj, t2, b + H + 4 * jj);
            }
            bar_wait<2 * T>(bar_pair);
            apply_g(b, gr);
            from_mid(b);  // b = dt1 (FIRST layout)
            const bool want_dx = p.dx != nullptr;
            DX* __restrict__ dxs = reinterpret_cast<DX*>(p.dx) + int64_t(s) * p.sample_elems + e0;
            for_each_vec<N, C, V_FIRST>(off_f, cmask, [&](auto m_, uint32_t off, uint32_t coord) {
                constexpr int m = decltype(m_)::value;
                const float4 q = raw4(stage_x, off);
                const float4 w = ldg4(s2p + coord);
                fma4(acc_2 + 4 * m, q, b + 4 * m);
                const float4 o = make_float4(q.x > relu_thr ? b[4 * m] * w.x : 0.f, q.y > relu_thr ? b[4 * m + 1] * w.y : 0.f,
                                             q.z > relu_thr ? b[4 * m + 2] * w.z : 0.f, q.w > relu_thr ? b[4 * m + 3] * w.w : 0.f);
                if (want_dx && (left >= TILE || off < left)) Io<DX>::st4(dxs + off, o);
            });
            mbar_arrive(&empty_bar[pair][st]);
        }
        for_each_vec<N, C, V_FIRST>(off_f, cmask, [&](auto m_, uint32_t off, uint32_t) {
            constexpr int m = decltype(m_)::value;
            *reinterpret_cast<float4*>(slab + 2 * TILE + off) = make_float4(acc_2[4 * m], acc_2[4 * m + 1], acc_2[4 * m + 2], acc_2[4 * m + 3]);
        });
        store_dg_half(acc_g, 1, slab);
    }
}

// ------------------------------------------------------------------ backward, TMEM edition (round 2)
// D >= 2048.  A three-view form of the kernel above is bound by the L1/shared-memory data pipe (77% of its peak at 48% of
// the HBM roofline, profiles/r01_bwd_notes.md item 7): ~3260 wavefronts per 4096-element tile pair, and because
// its single tile pair per SM runs all eight warps in lock-step, shared-memory phases and FP32 phases add up
// instead of overlapping.  Two views (64 floats per thread, ONE transposition per transform) need 1024 + 512
// (raw tiles) + 128 (dx) = 1664 wavefronts, but the round-1 attempt at it died of register pressure: 64 floats of
// stream + three 64-float running sums + three 64-float parameter vectors per thread.  Here everything that only
// its owner touches lives in TENSOR MEMORY instead (tmem.cuh: tcgen05.ld/st, 4-6x the bandwidth of shared
// memory and off its data path):
//   * the running sums ds1, ds2, dg (and dbias): load 32 columns, FFMA, store, once per tile;
//   * g (middle-layout order) and the Y role's s2;
//   * the X <-> Y exchange of half-streams (the "stash"): the X thread and the Y thread with the same tid sit in
//     warps w and w + 4, i.e. in the same TMEM lane, so one writes columns the other reads -- no shared memory.
// That leaves stream + one parameter vector in registers (no spills at 255), makes room for TWO tile pairs per
// SM at D <= 4096 (shared memory: 2 stages x (x, dy) + one in-place transposition buffer per role), and the two
// pairs are independent, so one pair's shared-memory phase overlaps the other's butterflies.
// TMEM columns per lane (E = 64 floats per thread, H = E / 2), shared by the X/Y thread pair of that lane:
//   [0,E) g | [E,2E) ds1 (X) | [2E,2E+H) dg lower half (X) | [2E+H,3E) dg upper half (Y) | [3E,4E) ds2 (Y) |
//   [4E,5E) s2 (Y) | [5E,5E+H) t2 upper half X->Y | [5E+H,6E) dt3 lower half Y->X | [6E,7E) the same for odd tiles |
//   [7E,8E) dbias (X)
// Everything else (bulk-copy staging ring, roles, workspace layout, second-stage reduction) is the kernel above.
template <int N, int C, int KT, int ROUNDS, bool WANT_DBIAS, bool RESID, class IO = float, class DX = IO>   // IO, DX: as above
__global__ void __launch_bounds__(256, 1) layer_bwd_tm_kernel(const BwdArgs p)
{
    static_assert(std::is_same_v<IO, float> || !RESID, "RESID (saved output + target) is fp32 only");
    constexpr int T = 1 << (N - C);
    constexpr int E = 1 << C;
    constexpr int H = E / 2;
    constexpr int PAIRS = 128 / T;
    constexpr int NS = 2;
    constexpr int64_t TILE = int64_t(1) << N;
    constexpr int SW = int(scratch_words(N, C));
    constexpr int PAIR_FLOATS = 2 * NS * int(TILE) + 2 * SW;
    static_assert(E == 64 && PAIRS >= 1 && PAIRS * T == 128, "layer_bwd_tm_kernel: 64 floats per thread, 4 warps per role");
    static_assert(ROUNDS == 3 || rounds_needed(N, C, N) <= 2, "2-view kernel needs FIRST+MID to cover all bits");
    static_assert(rounds_needed(N, C, N) <= 3, "FIRST+MID+LAST must cover every tile bit");
    // the exchange columns are double-buffered by tile parity (one pair barrier per tile instead of two)
    constexpr uint32_t COL_G = 0, COL_A1 = E, COL_AGX = 2 * E, COL_AGY = 2 * E + H, COL_A2 = 3 * E, COL_S2 = 4 * E,
                       COL_ST2 = 5 * E, COL_SD3 = 5 * E + H, COL_AB = 7 * E,   // ST2/SD3: + E * (tile & 1)
                       COL_PR = 7 * E;   // !WANT_DBIAS: this role's input-side parameter vector lives here, not in registers
    constexpr bool PR_TMEM = !WANT_DBIAS && !RESID;   // 64 fewer live registers: room for the scheduler to overlap the butterfly stages
    extern __shared__ float4 smem4[];
    __shared__ uint64_t full_bar[PAIRS][NS], empty_bar[PAIRS][NS];
    __shared__ uint64_t reads_done[PAIRS][2];   // per role: every thread has read the previous transposition out of the scratch
    __shared__ uint32_t tmem_base_smem;
    float* smem = reinterpret_cast<float*>(smem4);
    const int k = KT >= 0 ? KT : p.k;
    const uint32_t cmask = (1u << k) - 1u;
    const int s = blockIdx.x % p.n_samples;   // sample-minor CTA order
    const int cta_in_sample = blockIdx.x / p.n_samples;
    const int grp = s / p.spg;   // parameter group (Stacked block); the group's virtual samples read the inputs of samples 0 .. spg-1
    const IO* __restrict__ xbase = reinterpret_cast<const IO*>(p.x) + int64_t(s - grp * p.spg) * p.x_sample_stride;
    const float* __restrict__ s1p = p.s1 + int64_t(grp) * p.pstride;
    const float* __restrict__ s2p = p.s2 + int64_t(grp) * p.pstride;
    const IO* __restrict__ dybase = reinterpret_cast<const IO*>(p.dy) + int64_t(s) * p.sample_elems;

    if (threadIdx.x == 0) {
        for (int q = 0; q < PAIRS; ++q)
            for (int st = 0; st < NS; ++st) {
                mbar_init(&full_bar[q][st], 1);
                mbar_init(&empty_bar[q][st], 2 * T);
            }
        for (int q = 0; q < PAIRS; ++q) mbar_init(&reads_done[q][0], T), mbar_init(&reads_done[q][1], T);
        mbar_fence_init();
    }
    if (threadIdx.x < 32) tm_alloc(&tmem_base_smem, 512);
    tm_fence_before();
    __syncthreads();
    tm_fence_after();
    const uint32_t tm = tm_lane_base(tmem_base_smem);

    auto tile_of = [&](int it, int pr) -> int64_t {
        return ((int64_t(cta_in_sample) * p.iters_per_group + it) * PAIRS + pr) * TILE;
    };
    auto issue_tile = [&](int it, int pr) {
        if (it >= p.iters_per_group) return;
        const int64_t e0 = tile_of(it, pr);
        if (e0 >= p.sample_elems) return;
        const int st = it % NS;
        if (it >= NS) mbar_wait(&empty_bar[pr][st], ((it / NS) & 1) ^ 1);
        const int64_t left = p.sample_elems - e0;
        const uint32_t bytes = static_cast<uint32_t>((left < TILE ? left : TILE) * sizeof(IO));
        float* stage = smem + size_t(pr) * PAIR_FLOATS + size_t(st) * 2 * TILE;
        mbar_arrive_expect_tx(&full_bar[pr][st], 2 * bytes);
        bulk_g2s(stage, xbase + e0, bytes, &full_bar[pr][st]);
        bulk_g2s(stage + TILE, dybase + e0, bytes, &full_bar[pr][st]);
    };

    const int role = threadIdx.x / 128;               // 0 = X (warps 0..3), 1 = Y (warps 4..7): same TMEM quadrant per tid
    const int pair = (threadIdx.x % 128) / T;
    const uint32_t tid = threadIdx.x % T;
    float* pair_smem = smem + size_t(pair) * PAIR_FLOATS;
    float* scratch = pair_smem + 2 * NS * TILE + role * SW;   // this role's in-place transposition buffer
    const int bar_role = 1 + 3 * pair + role;
    const int bar_pair = 3 + 3 * pair;
    const float* __restrict__ gs = p.g + (int64_t(s) << k);
    float coef = 1.f;
    if constexpr (RESID) coef = __ldg(p.coef);
    const float dysc = p.dy_scale != nullptr ? __ldg(p.dy_scale) : 1.f;
    const float relu_thr = p.relu_in ? 0.f : -INFINITY;

    const uint32_t off_f = tile_thread_offset<N, C, V_FIRST>(tid);
    const uint32_t off_l = tile_thread_offset<N, C, V_LAST>(tid);
    const uint32_t wb_fm = transpose_writer_base<N, C, V_FIRST, V_MID>(tid);
    const uint32_t wb_ml = transpose_writer_base<N, C, V_MID, V_LAST>(tid);
    const uint32_t wb_lm = transpose_writer_base<N, C, V_LAST, V_MID2>(tid);
    const uint32_t wb_mf = ROUNDS == 3 ? transpose_writer_base<N, C, V_MID2, V_FIRST>(tid)
                                       : transpose_writer_base<N, C, V_MID, V_FIRST>(tid);
    const uint32_t mid_logical = view_tid_logical(view_mid(N, C), tid);

    int it_now = 0;
    const uint32_t col_acc = role ? COL_A2 : COL_A1;          // this role's end-product running sum
    auto to_mid = [&](float (&v)[E]) {
        if constexpr (ROUNDS == 3) {
            transform_in<N, C, KT, T, true>(v, scratch, scratch, tid, bar_role, k, wb_fm, wb_ml);
        } else {
            bfly_round<N, C, KT, SEQ2_IN, 0>(v, k);
            // the previous tile's second transposition has been read out by every thread of the role: an mbarrier
            // they arrived on right after those reads (a whole end-product section ago), not a blocking barrier
            if (it_now > 0) mbar_wait(&reads_done[pair][role], (it_now - 1) & 1);
            transpose_write<N, C, V_FIRST, V_MID>(v, scratch, wb_fm);
            role_sync<T>(bar_role);
            transpose_read<C>(v, scratch, tid);
            bfly_round<N, C, KT, SEQ2_IN, 1>(v, k);
        }
    };
    auto from_mid = [&](float (&v)[E], float* acc_lo) {
        if constexpr (ROUNDS == 3) {
            transform_out<N, C, KT, T, true>(v, scratch, scratch, tid, bar_role, k, wb_lm, wb_mf);
            tm_ld32(acc_lo, tm + col_acc);
        } else {
            bfly_round<N, C, KT, SEQ2_OUT, 0>(v, k);
            // no barrier before the write: the pair barrier of the half-stream exchange lies between the first
            // transposition's reads and this write
            transpose_write<N, C, V_MID, V_FIRST>(v, scratch, wb_mf);
            role_sync<T>(bar_role);
            transpose_read<C>(v, scratch, tid);
            mbar_arrive(&reads_done[pair][role]);
            tm_ld32(acc_lo, tm + col_acc);   // the end product's first running-sum chunk: in flight during the butterflies
            bfly_round<N, C, KT, SEQ2_OUT, 1>(v, k);
        }
    };
    // v *= g: g comes from TMEM in the middle layout's register order, 32 columns at a time
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
    auto store_dg_half = [&](const float* acc, int half_is_upper, float* dst) {
        if constexpr (ROUNDS == 3) {
            for_each_vec<N, C, V_LAST>(off_l, cmask, [&](auto m_, uint32_t off, uint32_t) {
                constexpr int m = decltype(m_)::value;
                constexpr int mh = m % (E / 8);
                if ((m >= E / 8) == (half_is_upper != 0))
                    *reinterpret_cast<float4*>(dst + off) = make_float4(acc[4 * mh], acc[4 * mh + 1], acc[4 * mh + 2], acc[4 * mh + 3]);
            });
        } else {
            static_for<0, E / 2>([&](auto r_) {
                constexpr int r = decltype(r_)::value;
                constexpr uint32_t rl_lo = view_reg_logical(view_mid(N, C), r);
                constexpr uint32_t rl_hi = view_reg_logical(view_mid(N, C), r + E / 2);
                dst[mid_logical | (half_is_upper ? rl_hi : rl_lo)] = acc[r];
            });
        }
    };
    float* __restrict__ slab = p.ws + (((int64_t(s) * p.ctas_per_sample + cta_in_sample) * PAIRS + pair) * 4) * TILE;

    auto zero_tail = [&](float* stage_x, int64_t left) {
        if (left < TILE) {
            static_for<0, E / 4>([&](auto m_) {
                constexpr int m = decltype(m_)::value;
                const uint32_t off = off_f + tile_reg_offset<N, C, V_FIRST>(m);
                if (off >= left) {
                    Io<IO>::sts_zero4(reinterpret_cast<IO*>(stage_x) + off);
                    Io<IO>::sts_zero4(reinterpret_cast<IO*>(stage_x + TILE) + off);
                }
            });
        }
    };
    auto raw4 = [&](const float* stage_tile, uint32_t off) -> float4 {
        return Io<IO>::lds4(reinterpret_cast<const IO*>(stage_tile) + off);
    };
    // RESID: dy = coef * (saved output - target); the target (shared by all samples, L2-resident) is read from
    // global memory, zero beyond the valid part of a partial tile
    auto to_dy = [&](float4 q, const float* tgt, uint32_t off, int64_t left) -> float4 {
        if constexpr (RESID) {
            float4 tg = make_float4(0.f, 0.f, 0.f, 0.f);
            if (left >= TILE || off < left) tg = ldg4(tgt + off);
            q = make_float4(coef * (q.x - tg.x), coef * (q.y - tg.y), coef * (q.z - tg.z), coef * (q.w - tg.w));
        } else {
            q = make_float4(dysc * q.x, dysc * q.y, dysc * q.z, dysc * q.w);
        }
        return q;
    };

    // ---- TMEM initialisation: running sums = 0; g (X writes it, both roles read it); s2 (Y)
    {
        float z[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) z[i] = 0.f;
        if (role == 0) {
            tm_st32(z, tm + COL_A1), tm_st32(z, tm + COL_A1 + 32), tm_st32(z, tm + COL_AGX);
            if constexpr (WANT_DBIAS) tm_st32(z, tm + COL_AB), tm_st32(z, tm + COL_AB + 32);
            float gr[E];
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
            tm_st32(gr, tm + COL_G), tm_st32(gr + 32, tm + COL_G + 32);
        } else {
            tm_st32(z, tm + COL_A2), tm_st32(z, tm + COL_A2 + 32), tm_st32(z, tm + COL_AGY);
            float sr[E];
            for_each_vec<N, C, V_FIRST>(off_f, cmask, [&](auto m_, uint32_t, uint32_t coord) {
                constexpr int m = decltype(m_)::value;
                const float4 w = ldg4(s2p + coord);
                sr[4 * m] = w.x, sr[4 * m + 1] = w.y, sr[4 * m + 2] = w.z, sr[4 * m + 3] = w.w;
            });
            tm_st32(sr, tm + COL_S2), tm_st32(sr + 32, tm + COL_S2 + 32);
        }
        tm_wait_st();
        tm_fence_before();
        __syncthreads();
        tm_fence_after();
    }

    // ONE instruction stream for both roles (the two transforms, the g multiply, the running-sum updates are the same
    // code on different data; only the half-stream exchange and the dx store are role-specific): the fully unrolled
    // 64-float transforms are ~8 KB of SASS each, and with a private copy per role the hot loop (53 KB) thrashed the
    // 32 KB instruction cache -- "no instruction" was the top stall reason (22% of samples, profiles/r02_bwd_notes.md).
    //   X: v = s2 * x  -> t2  -> t4,   end product ds1 += dy * t4 (dbias += dy)
    //   Y: v = s1 * dy -> dt3 -> dt1,  end product ds2 += x * dt1, dx = s2 * dt1
    float pr[PR_TMEM ? 1 : E];   // this role's input-side parameter vector: X s2, Y s1 (FIRST-view order)
    {
        // the upstream gradient is dy_scale * dy: folded into Y's s1 once (s1 * dy_scale) and into X's sums at the end
        // (ds1, dbias are linear in dy), not applied to every element of every tile
        const float* __restrict__ pv = role ? s1p : s2p;
        const float psc = (!RESID && role) ? dysc : 1.f;
        float w[E];
        for_each_vec<N, C, V_FIRST>(off_f, cmask, [&](auto m_, uint32_t, uint32_t coord) {
            constexpr int m = decltype(m_)::value;
            const float4 q = ldg4(pv + coord);
            w[4 * m] = psc * q.x, w[4 * m + 1] = psc * q.y, w[4 * m + 2] = psc * q.z, w[4 * m + 3] = psc * q.w;
        });
        if constexpr (PR_TMEM) {
            // Y's s1 * dy_scale goes to COL_PR; X's vector is s2, which Y already keeps in COL_S2 of the same lane
            if (role) {
                tm_st32(w, tm + COL_PR), tm_st32(w + 32, tm + COL_PR + 32);
                tm_wait_st();
            }
        } else {
#pragma unroll
            for (int i = 0; i < E; ++i) pr[i] = w[i];
        }
    }
    const uint32_t col_pr = role ? COL_PR : COL_S2;
    if (role == 0 && tid == 0)
        for (int i = 0; i < NS - 1; ++i) issue_tile(i, pair);
#pragma unroll 1
    for (int it = 0; it < p.iters_per_group; ++it) {
        const int64_t e0 = tile_of(it, pair);
        if (e0 >= p.sample_elems) break;
        const int64_t left = p.sample_elems - e0;
        const int st = it % NS;
        float* stage_x = pair_smem + size_t(st) * 2 * TILE;
        const float* stage_dy = stage_x + TILE;
        const float* tgt = RESID ? p.target + e0 : nullptr;
        const float* src_in = role ? stage_dy : stage_x;       // the stream this role transforms
        const float* src_end = role ? stage_x : stage_dy;      // the other raw tile, for the end product
        if (role == 0 && tid == 0) issue_tile(it + NS - 1, pair);
        mbar_wait(&full_bar[pair][st], (it / NS) & 1);
        zero_tail(stage_x, left);
        float v[E];
        if constexpr (RESID) {
            if (role) {
                for_each_vec<N, C, V_FIRST>(off_f, cmask, [&](auto m_, uint32_t off, uint32_t) {
                    constexpr int m = decltype(m_)::value;
                    mul4(v + 4 * m, to_dy(raw4(stage_dy, off), tgt, off, left), make_float4(pr[4 * m], pr[4 * m + 1], pr[4 * m + 2], pr[4 * m + 3]));
                });
            } else {
                for_each_vec<N, C, V_FIRST>(off_f, cmask, [&](auto m_, uint32_t off, uint32_t) {
                    constexpr int m = decltype(m_)::value;
                    mul4(v + 4 * m, raw4(stage_x, off), make_float4(pr[4 * m], pr[4 * m + 1], pr[4 * m + 2], pr[4 * m + 3]));
                });
            }
        } else if constexpr (PR_TMEM) {
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                float w[32];
                tm_ld32(w, tm + col_pr + 32 * c);
                float4 q[8];
                static_for<0, 8>([&](auto j_) {
                    constexpr int j = decltype(j_)::value;
                    q[j] = raw4(src_in, off_f + tile_reg_offset<N, C, V_FIRST>(8 * c + j));
                });
                tm_wait_ld();
#pragma unroll
                for (int j = 0; j < 8; ++j) mul4(v + 32 * c + 4 * j, q[j], make_float4(w[4 * j], w[4 * j + 1], w[4 * j + 2], w[4 * j + 3]));
            }
        } else {
            for_each_vec<N, C, V_FIRST>(off_f, cmask, [&](auto m_, uint32_t off, uint32_t) {
                constexpr int m = decltype(m_)::value;
                mul4(v + 4 * m, raw4(src_in, off), make_float4(pr[4 * m], pr[4 * m + 1], pr[4 * m + 2], pr[4 * m + 3]));
            });
        }
        it_now = it;
        to_mid(v);  // X: t2, Y: dt3 (middle layout)
        // half-stream exchange through TMEM: X publishes the upper half of t2 and accumulates the lower half of dg,
        // Y publishes the lower half of dt3 and accumulates the upper half.  Columns alternate with the tile parity,
        // so ONE pair barrier per tile suffices: a thread overwrites buffer p two tiles later, after the barrier of the
        // tile in between, which its partner only reaches after it has read buffer p.
        const uint32_t par = uint32_t(it & 1) * E;
        if (role == 0) tm_st32(v + H, tm + COL_ST2 + par); else tm_st32(v, tm + COL_SD3 + par);
        tm_wait_st();
        tm_fence_before();
        bar_wait<2 * T>(bar_pair);
        tm_fence_after();
        {
            float oth[H], ag[H];
            tm_ld32(oth, tm + (role ? COL_ST2 : COL_SD3) + par);
            tm_ld32(ag, tm + (role ? COL_AGY : COL_AGX));
            tm_wait_ld();
            if (role == 0) {
#pragma unroll
                for (int jj = 0; jj < H / 4; ++jj)
                    fma4(ag + 4 * jj, make_float4(oth[4 * jj], oth[4 * jj + 1], oth[4 * jj + 2], oth[4 * jj + 3]), v + 4 * jj);
            } else {
#pragma unroll
                for (int jj = 0; jj < H / 4; ++jj)
                    fma4(ag + 4 * jj, make_float4(oth[4 * jj], oth[4 * jj + 1], oth[4 * jj + 2], oth[4 * jj + 3]), v + H + 4 * jj);
            }
            tm_st32(ag, tm + (role ? COL_AGY : COL_AGX));
        }
        apply_g(v);
        float acc0[32];
        from_mid(v, acc0);  // X: t4, Y: dt1 (FIRST layout); acc0 = running-sum chunk 0, load in flight
        const bool want_dx = p.dx != nullptr;
        DX* __restrict__ dxs = reinterpret_cast<DX*>(p.dx) + int64_t(s) * p.sample_elems + e0;
#pragma unroll
        for (int c = 0; c < 2; ++c) {   // end product, 32 registers at a time
            float acc1[32];
            float* acc = c == 0 ? acc0 : acc1;
            if (c == 1) tm_ld32(acc1, tm + col_acc + 32);
            float4 q[8];
            if constexpr (RESID) {
                if (role == 0) {
                    static_for<0, 8>([&](auto j_) {
                        constexpr int j = decltype(j_)::value;
                        const uint32_t off = off_f + tile_reg_offset<N, C, V_FIRST>(8 * c + j);
                        q[j] = to_dy(raw4(stage_dy, off), tgt, off, left);
                    });
                } else {
                    static_for<0, 8>([&](auto j_) {
                        constexpr int j = decltype(j_)::value;
                        q[j] = raw4(stage_x, off_f + tile_reg_offset<N, C, V_FIRST>(8 * c + j));
                    });
                }
            } else {
                static_for<0, 8>([&](auto j_) {
                    constexpr int j = decltype(j_)::value;
                    q[j] = raw4(src_end, off_f + tile_reg_offset<N, C, V_FIRST>(8 * c + j));
                });
            }
            tm_wait_ld();
#pragma unroll
            for (int j = 0; j < 8; ++j) fma4(acc + 4 * j, q[j], v + 32 * c + 4 * j);
            tm_st32(acc, tm + col_acc + 32 * c);
            if (role) {   // dx = s2 * dt1, masked by the fused ReLU of the producer
                float w[32];
                tm_ld32(w, tm + COL_S2 + 32 * c);
                tm_wait_ld();
                static_for<0, 8>([&](auto j_) {
                    constexpr int j = decltype(j_)::value;
                    const uint32_t off = off_f + tile_reg_offset<N, C, V_FIRST>(8 * c + j);
                    const float* bb = v + 32 * c + 4 * j;
                    const float4 o = make_float4(q[j].x > relu_thr ? bb[0] * w[4 * j] : 0.f, q[j].y > relu_thr ? bb[1] * w[4 * j + 1] : 0.f,
                                                 q[j].z > relu_thr ? bb[2] * w[4 * j + 2] : 0.f, q[j].w > relu_thr ? bb[3] * w[4 * j + 3] : 0.f);
                    if (want_dx && (left >= TILE || off < left)) Io<DX>::st4(dxs + off, o);
                });
            } else if constexpr (WANT_DBIAS) {
                float ab[32];
                tm_ld32(ab, tm + COL_AB + 32 * c);
                tm_wait_ld();
#pragma unroll
                for (int j = 0; j < 8; ++j) ab[4 * j] += q[j].x, ab[4 * j + 1] += q[j].y, ab[4 * j + 2] += q[j].z, ab[4 * j + 3] += q[j].w;
                tm_st32(ab, tm + COL_AB + 32 * c);
            }
        }
        mbar_arrive(&empty_bar[pair][st]);
        tm_wait_st();   // this thread's next loads of the running sums come after these stores
    }
    // running sums -> workspace: [0] dg, [1] ds1, [2] ds2, [3] dbias
#pragma unroll
    for (int c = 0; c < 2; ++c) {
        float acc[32];
        tm_ld32(acc, tm + col_acc + 32 * c);
        tm_wait_ld();
        float* dst = slab + (role ? 2 : 1) * TILE;
        const float osc = (RESID || role) ? 1.f : dysc;   // X: ds1 = dy_scale * sum dy * t4
        static_for<0, 8>([&](auto j_) {
            constexpr int j = decltype(j_)::value;
            const uint32_t off = off_f + tile_reg_offset<N, C, V_FIRST>(8 * c + j);
            *reinterpret_cast<float4*>(dst + off) = make_float4(osc * acc[4 * j], osc * acc[4 * j + 1], osc * acc[4 * j + 2], osc * acc[4 * j + 3]);
        });
        if constexpr (WANT_DBIAS) {
            if (role == 0) {
                tm_ld32(acc, tm + COL_AB + 32 * c);
                tm_wait_ld();
                static_for<0, 8>([&](auto j_) {
                    constexpr int j = decltype(j_)::value;
                    const uint32_t off = off_f + tile_reg_offset<N, C, V_FIRST>(8 * c + j);
                    *reinterpret_cast<float4*>(slab + 3 * TILE + off) = make_float4(osc * acc[4 * j], osc * acc[4 * j + 1], osc * acc[4 * j + 2], osc * acc[4 * j + 3]);
                });
            }
        }
    }
    {
        float ag[H];
        tm_ld32(ag, tm + (role ? COL_AGY : COL_AGX));
        tm_wait_ld();
        store_dg_half(ag, role, slab);
    }
    tm_fence_before();
    __syncthreads();
    if (threadIdx.x < 32) tm_dealloc(tmem_base_smem, 512);
}

// Second stage: fixed-order (bit-reproducible, no atomics) sums of the per-group slabs.
//   dg[s, i]         = sum over the slabs of sample s and over the N/D row replicas inside a slab
//   ds1/ds2/dbias[i] = the same over ALL slabs
// Workspace layout: [slab][quantity 0..3 = dg, ds1, ds2, dbias][tile element], slabs sample-major.
//
// Pass A (layer_bwd_reduce_slabs_kernel): one thread per (sample, quantity, float4 of the tile)
// adds up that sample's slabs -- consecutive threads read consecutive addresses, so the whole
// workspace streams through once at L2/HBM speed -- and leaves the sum in the sample's first slab
// (in place: a thread only ever touches its own column).  With one row per tile (D == tile) the
// dg sums go straight to their destination.
// Pass B (layer_bwd_reduce_fold_kernel): one warp per output coordinate folds the row replicas
// (dg) or the replicas and samples (ds1, ds2, dbias) of the S per-sample sums: a few MB, L2-resident.
__global__ void __launch_bounds__(256)
layer_bwd_reduce_slabs_kernel(float* __restrict__ ws, float* __restrict__ dg_direct, int S, int slabs_per_sample, int64_t tile4)
{
    const int64_t e = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;  // float4 index inside the tile
    if (e >= tile4) return;
    const int q = blockIdx.y;
    const int64_t stride = 4 * tile4;
    for (int s = blockIdx.z; s < S; s += gridDim.z) {
    float4* base = reinterpret_cast<float4*>(ws) + (int64_t(s) * slabs_per_sample * 4 + q) * tile4 + e;
    float4 acc = base[0];
    int j = 1;
    for (; j + 4 <= slabs_per_sample; j += 4) {  // four independent loads in flight, added in slab order
        const float4 a0 = base[(j + 0) * stride], a1 = base[(j + 1) * stride], a2 = base[(j + 2) * stride],
                     a3 = base[(j + 3) * stride];
        acc.x = (((acc.x + a0.x) + a1.x) + a2.x) + a3.x;
        acc.y = (((acc.y + a0.y) + a1.y) + a2.y) + a3.y;
        acc.z = (((acc.z + a0.z) + a1.z) + a2.z) + a3.z;
        acc.w = (((acc.w + a0.w) + a1.w) + a2.w) + a3.w;
    }
    for (; j < slabs_per_sample; ++j) {
        const float4 a0 = base[j * stride];
        acc.x += a0.x, acc.y += a0.y, acc.z += a0.z, acc.w += a0.w;
    }
    if (q == 0 && dg_direct)
        reinterpret_cast<float4*>(dg_direct)[int64_t(s) * tile4 + e] = acc;
    else
        base[0] = acc;
    }
}

__global__ void __launch_bounds__(256)
layer_bwd_reduce_fold_kernel(const float* __restrict__ ws, float* __restrict__ dg, float* __restrict__ ds1,
                             float* __restrict__ ds2, float* __restrict__ dbias, int S, int slabs_per_sample, int64_t tile, int D,
                             int dg_blocks, int cta_per_output, int groups)
{
    __shared__ float red[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int reps = static_cast<int>(tile / D);
    const int64_t sample_stride = int64_t(slabs_per_sample) * 4 * tile;  // first slab of sample s
    const unsigned full = 0xffffffffu;
    const int nq = dbias ? 3 : 2;
    if (static_cast<int>(blockIdx.x) < dg_blocks) {  // dg: one warp per (sample, coordinate), `reps` terms
        const int64_t w = int64_t(blockIdx.x) * 8 + warp;
        if (w >= int64_t(S) * D) return;
        const int s = static_cast<int>(w / D), i = static_cast<int>(w % D);
        const float* base = ws + s * sample_stride + i;
        float acc = 0.f;
        for (int r = lane; r < reps; r += 32) acc += base[int64_t(r) * D];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(full, acc, o);
        if (lane == 0) dg[w] = acc;
        return;
    }
    // ds1, ds2, dbias: S * reps terms per coordinate; a whole CTA per output when that is many
    const int64_t o = cta_per_output ? int64_t(blockIdx.x) - dg_blocks : (int64_t(blockIdx.x) - dg_blocks) * 8 + warp;
    const int64_t GD = int64_t(groups) * D;   // grouped launch: one (D) output vector per parameter group, over that group's samples
    if (o >= int64_t(nq) * GD) return;
    const int q = 1 + static_cast<int>(o / GD), gi = static_cast<int>(o % GD), grp = gi / D, i = gi - grp * D;
    const int spg = S / groups;
    const float* base = ws + int64_t(q) * tile + i + int64_t(grp) * spg * sample_stride;
    const int terms = spg * reps;
    const int first = cta_per_output ? threadIdx.x : lane, step = cta_per_output ? 256 : 32;
    float acc = 0.f;
#pragma unroll 4
    for (int t = first; t < terms; t += step) acc += base[(t / reps) * sample_stride + int64_t(t % reps) * D];
#pragma unroll
    for (int sh = 16; sh > 0; sh >>= 1) acc += __shfl_xor_sync(full, acc, sh);
    if (cta_per_output) {
        if (lane == 0) red[warp] = acc;
        __syncthreads();
        if (threadIdx.x != 0) return;
        acc = red[0];
#pragma unroll
        for (int j = 1; j < 8; ++j) acc += red[j];
    } else if (lane != 0) {
        return;
    }
    (q == 1 ? ds1 : q == 2 ? ds2 : dbias)[gi] = acc;
}

int launch_bwd_reduce(float* ws, float* dg, float* ds1, float* ds2, float* dbias, int64_t S, int slabs_per_sample,
                      int64_t tile, int64_t D, cudaStream_t stream, int64_t groups)
{
    const int64_t tile4 = tile / 4;
    const bool direct = D == tile;  // one row per tile: pass A's dg sums are final
    if (slabs_per_sample > 1 || direct) {
        dim3 agrid(static_cast<unsigned>((tile4 + 255) / 256), dbias ? 4u : 3u, static_cast<unsigned>(S > 65535 ? 65535 : S));
        layer_bwd_reduce_slabs_kernel<<<agrid, 256, 0, stream>>>(ws, direct ? dg : nullptr, static_cast<int>(S), slabs_per_sample, tile4);
        if (int rc = check_launch("layer_bwd_reduce_slabs_kernel")) return rc;
    }
    const int64_t dg_blocks = direct ? 0 : (S * D + 7) / 8;
    const int64_t ds_outputs = (dbias ? 3 : 2) * D * groups;
    const int cta_per_output = (S / groups) * (tile / D) >= 1024;
    const int64_t ds_blocks = cta_per_output ? ds_outputs : (ds_outputs + 7) / 8;
    layer_bwd_reduce_fold_kernel<<<static_cast<unsigned>(dg_blocks + ds_blocks), 256, 0, stream>>>(
        ws, dg, ds1, ds2, dbias, static_cast<int>(S), slabs_per_sample, tile, static_cast<int>(D), static_cast<int>(dg_blocks),
        cta_per_output, static_cast<int>(groups));
    return check_launch("layer_bwd_reduce_fold_kernel");
}

template <int N, int C, int KT>
static int launch_bwd_tma_cfg(const LayerBwdCall& c, int k, cudaStream_t stream)
{
    static unsigned char smem_ok[8][64] = {};
    constexpr int T = 1 << (N - C);
    constexpr int PAIRS = 128 / T;
    constexpr size_t tile = size_t(1) << N;
    constexpr size_t sw = scratch_words(N, C);
    constexpr size_t smem_plain = bwd_smem_bytes(N, PAIRS, 2, sw);
    constexpr size_t smem_tgt = bwd_smem_bytes(N, PAIRS, 3, sw);  // RESID with the target staged
    static_assert(smem_plain <= 227 * 1024, "backward kernel shared memory");
    const size_t smem = (c.target != nullptr && bwd_stage_target(N, PAIRS, sw)) ? smem_tgt : smem_plain;
    const int64_t D = int64_t(1) << k;
    const int64_t tiles_per_sample = (c.B * D + int64_t(tile) - 1) / int64_t(tile);
    const Plan plan = make_plan_waves(c.S, tiles_per_sample, PAIRS, 148, 8, 8);
    const size_t need = sizeof(float) * size_t(c.S) * plan.ctas_per_sample * PAIRS * 4 * tile;
    if (c.need_only) {
        *c.need_only = need;
        return WHVI_OK;
    }
    if (c.ws == nullptr || c.ws_bytes < need)
        return fail(WHVI_E_WORKSPACE, "layer_bwd: workspace of %zu bytes needed, %zu given", need, c.ws_bytes);
    const int64_t ctas = int64_t(plan.ctas_per_sample) * c.S;
    if (ctas > 0x7fffffffLL) return fail(WHVI_E_SHAPE, "layer_bwd: grid too large");
    BwdArgs a{c.x, c.xs, c.dy, c.g, c.s1, c.s2, c.dx, c.ws, c.B * D, static_cast<int>(c.S), plan.ctas_per_sample, plan.iters_per_group, k,
              c.relu_in, c.target, c.coef, c.dy_scale};
    a.spg = static_cast<int>(c.S / c.groups);
    a.pstride = static_cast<int>(c.pstride);
    auto go = [&](auto kernel, int slot) -> int {
        if (int rc = ensure_smem(kernel, smem, smem_ok[slot])) return rc;
        kernel<<<static_cast<unsigned>(ctas), 256, smem, stream>>>(a);
        return check_launch("layer_bwd_tma_kernel");
    };
    const bool db = c.dbias != nullptr, rs = c.target != nullptr;
    int rc;
    if (c.bf16) {
        if (rs) return fail(WHVI_E_MODE, "layer_bwd: bf16 activations cannot be combined with a target");
        if (c.dx_f32)
            rc = db ? go(layer_bwd_tma_kernel<N, C, KT, true, false, __nv_bfloat16, float>, 6)
                    : go(layer_bwd_tma_kernel<N, C, KT, false, false, __nv_bfloat16, float>, 7);
        else rc = db ? go(layer_bwd_tma_kernel<N, C, KT, true, false, __nv_bfloat16>, 4)
                     : go(layer_bwd_tma_kernel<N, C, KT, false, false, __nv_bfloat16>, 5);
    } else if (db && rs) rc = go(layer_bwd_tma_kernel<N, C, KT, true, true>, 0);
    else if (db) rc = go(layer_bwd_tma_kernel<N, C, KT, true, false>, 1);
    else if (rs) rc = go(layer_bwd_tma_kernel<N, C, KT, false, true>, 2);
    else rc = go(layer_bwd_tma_kernel<N, C, KT, false, false>, 3);
    if (rc) return rc;
    return launch_bwd_reduce(c.ws, c.dg, c.ds1, c.ds2, c.dbias, c.S, plan.ctas_per_sample * PAIRS, int64_t(tile), D, stream, c.groups);
}

template <int N, int C, int KT, int ROUNDS>
static int launch_bwd_tm_cfg(const LayerBwdCall& c, int k, cudaStream_t stream)
{
    static unsigned char smem_ok[8][64] = {};
    constexpr int T = 1 << (N - C);
    constexpr int PAIRS = 128 / T;
    constexpr size_t tile = size_t(1) << N;
    constexpr size_t smem = sizeof(float) * PAIRS * (2 * 2 * tile + 2 * size_t(scratch_words(N, C)));
    static_assert(smem <= 227 * 1024, "TMEM backward kernel shared memory");
    const int64_t D = int64_t(1) << k;
    const int64_t tiles_per_sample = (c.B * D + int64_t(tile) - 1) / int64_t(tile);
    const Plan plan = make_plan_waves(c.S, tiles_per_sample, PAIRS, 148, 8, 8);
    const size_t need = sizeof(float) * size_t(c.S) * plan.ctas_per_sample * PAIRS * 4 * tile;
    if (c.need_only) {
        *c.need_only = need;
        return WHVI_OK;
    }
    if (c.ws == nullptr || c.ws_bytes < need)
        return fail(WHVI_E_WORKSPACE, "layer_bwd: workspace of %zu bytes needed, %zu given", need, c.ws_bytes);
    const int64_t ctas = int64_t(plan.ctas_per_sample) * c.S;
    if (ctas > 0x7fffffffLL) return fail(WHVI_E_SHAPE, "layer_bwd: grid too large");
    BwdArgs a{c.x, c.xs, c.dy, c.g, c.s1, c.s2, c.dx, c.ws, c.B * D, static_cast<int>(c.S), plan.ctas_per_sample, plan.iters_per_group, k,
              c.relu_in, c.target, c.coef, c.dy_scale};
    a.spg = static_cast<int>(c.S / c.groups);
    a.pstride = static_cast<int>(c.pstride);
    auto go = [&](auto kernel, int slot) -> int {
        if (int rc = ensure_smem(kernel, smem, smem_ok[slot])) return rc;
        kernel<<<static_cast<unsigned>(ctas), 256, smem, stream>>>(a);
        return check_launch("layer_bwd_tm_kernel");
    };
    const bool db = c.dbias != nullptr, rs = c.target != nullptr;
    int rc;
    if (c.bf16) {
        if (rs) return fail(WHVI_E_MODE, "layer_bwd: bf16 activations cannot be combined with a target");
        if (c.dx_f32)
            rc = db ? go(layer_bwd_tm_kernel<N, C, KT, ROUNDS, true, false, __nv_bfloat16, float>, 6)
                    : go(layer_bwd_tm_kernel<N, C, KT, ROUNDS, false, false, __nv_bfloat16, float>, 7);
        else rc = db ? go(layer_bwd_tm_kernel<N, C, KT, ROUNDS, true, false, __nv_bfloat16>, 4)
                     : go(layer_bwd_tm_kernel<N, C, KT, ROUNDS, false, false, __nv_bfloat16>, 5);
    } else if (db && rs) rc = go(layer_bwd_tm_kernel<N, C, KT, ROUNDS, true, true>, 0);
    else if (db) rc = go(layer_bwd_tm_kernel<N, C, KT, ROUNDS, true, false>, 1);
    else if (rs) rc = go(layer_bwd_tm_kernel<N, C, KT, ROUNDS, false, true>, 2);
    else rc = go(layer_bwd_tm_kernel<N, C, KT, ROUNDS, false, false>, 3);
    if (rc) return rc;
    return launch_bwd_reduce(c.ws, c.dg, c.ds1, c.ds2, c.dbias, c.S, plan.ctas_per_sample * PAIRS, int64_t(tile), D, stream, c.groups);
}

int launch_layer_bwd(const LayerBwdCall& c, int64_t D, cudaStream_t stream)
{
    const int k = ilog2(D);
    // D <= 1024: TMA-staged kernels, one CTA per SM, NS = 2 stages, ping-pong transposition buffers, parameters
    // register-resident, two views (FIRST + MID cover all 10 tile bits), one warp per role, 4 pairs per CTA
    if (k >= 2 && k <= 6) return launch_bwd_tma_cfg<10, 5, k_family(2, 6)>(c, k, stream);
    if (k >= 7 && k <= 9) return launch_bwd_tma_cfg<10, 5, k_family(7, 9)>(c, k, stream);
    if (k == 10) return launch_bwd_tma_cfg<10, 5, 10>(c, k, stream);
    // D = 2048, 4096: two views, 64 floats per thread, running sums / g / role exchange in tensor memory
    if (k == 11) return launch_bwd_tm_cfg<12, 6, 11, 2>(c, k, stream);
    if (k == 12) return launch_bwd_tm_cfg<12, 6, 12, 2>(c, k, stream);
    // D = 8192: three views, 64 floats per thread, one tile pair per CTA, same tensor-memory residency
    if (k == 13) return launch_bwd_tm_cfg<13, 6, 13, 3>(c, k, stream);
    return fail(WHVI_E_SHAPE, "layer_bwd: D = %lld unsupported (4 <= D <= 8192)", (long long)D);
}

}  // namespace whvi
