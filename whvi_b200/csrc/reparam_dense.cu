// Kernel (4), dense form: the reparameterisation with a full lower-triangular covariance factor and its backward as
// hand-written tcgen05 tensor-core GEMMs, plus kernel (5) for that posterior: the Gaussian KL with its log-determinant.
//
//   forward   G[s, i] = mu[i] + sum_{j <= i} L[i, j] E[s, j]                 (D x D times D x S: "a dense contraction over MC samples")
//   backward  dL[i, j] = sum_s dG[s, i] E[s, j]  for j <= i, 0 above         (D x S times S x D)
//   KL        0.5 ( D ln(lambda) - 2 sum ln L_ii - D + |L|_F^2 / lambda + |mu|^2 / lambda ),  dL = L / lambda - diag(1 / L_ii)
//
// The reference's posterior is diagonal (g = mu + softplus(rho) * eps, src/weights.py:43-50, :82-83; SURVEY F5); this is
// the north-star's superset.  Not in the reference => no reference golden ("parity unpinned"); the oracle is the fp64
// formula (oracle_reparam(dense=1), numpy for dL and the KL).
//
// One warp-specialised GEMM kernel serves both products (C[m, n] = sum_k A[m, k] B[n, k], A and B K-major):
//   warp 0    TMA producer: cp.async.bulk.tensor.2d of a 128 x 32 fp32 box of A and an N x 32 box of B per K block into
//             128-byte-swizzled shared-memory tiles, mbarrier transaction counts (UTMALDG in SASS);
//   warps 2-5 operand split: fp32 accuracy on tf32 hardware needs x = hi + lo.  The tensor core ignores the low 13
//             mantissa bits of a tf32 operand, so the RAW tile is the hi operand as it lies; these warps only compute
//             lo = x - trunc(x) into a second tile with the same swizzle (and zero the entries above the diagonal of
//             the triangular operand in the blocks that straddle it);
//   warp 1    one thread issues tcgen05.mma kind::tf32 (M = 128, N <= 256, K = 8): hi*hi + hi*lo + lo*hi into the TMEM
//             accumulator (the dropped lo*lo term is ~2^-22 relative), tcgen05.commit frees the stage;
//   warps 2-5 epilogue: tcgen05.ld (lane = row m), coalesced stores.
// Work split: the forward is a triangle (row block rb has rb + 1 column blocks), so one CTA per row block (round 1:
// 32 CTAs, the last 32 times longer than the first) leaves the chip idle.  Here a work unit is (row block, chunk of
// q column blocks): ~148 units of equal size at D = 4096, partial accumulators go to a workspace and a second kernel
// adds them in a fixed order (bit-reproducible) together with mu.
#include <cuda.h>
#include "common.cuh"
#include "engine.cuh"
#include "tmem.cuh"

namespace whvi {

constexpr int DG_BM = 128;        // rows of A per unit = TMEM lanes
constexpr int DG_BK = 32;         // fp32 per K block = one 128-byte swizzle row
constexpr int DG_THREADS = 192;   // producer warp, MMA warp, four split/epilogue warps
constexpr int DG_TILE_A = DG_BM * DG_BK * 4;   // bytes

// ---- descriptors -------------------------------------------------------------------------------------------------
// cute::UMMA::SmemDescriptor, K-major SWIZZLE_128B: start >> 4 [0,14), LBO = 1 [16,30) (ignored for swizzled K-major),
// SBO = 1024 B >> 4 [32,46) (stride between 8-row groups), version = 1 [46,48), layout_type = 2 [61,64)
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr)
{
    return uint64_t((smem_addr >> 4) & 0x3FFFu) | (uint64_t(1) << 16) | (uint64_t(1024 >> 4) << 32) | (uint64_t(1) << 46) |
           (uint64_t(2) << 61);
}
// cute::UMMA::InstrDescriptor: c_format F32 = 1 [4,6), a/b_format TF32 = 2 [7,10) [10,13), a/b K-major [15],[16] = 0,
// n >> 3 [17,23), m >> 4 [24,29)
__device__ __forceinline__ uint32_t umma_idesc_tf32(int m, int n)
{
    return (1u << 4) | (2u << 7) | (2u << 10) | (uint32_t(n >> 3) << 17) | (uint32_t(m >> 4) << 24);
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
                 : "memory");
}

struct DenseGemmArgs {
    int mode;            // 0: reparameterisation (triangular A = L, split-K units), 1: outer product dL (lower-triangular tile pairs)
    int n;               // B rows per unit (MMA N): samples padded to 16 (mode 0), 128 (mode 1)
    int q;               // mode 0: column blocks (of 128) per work unit
    int k_blocks_total;  // mode 1: K blocks (of 32) of the contraction
    int D;
    int S;               // mode 0: valid samples (<= n)
    const float* mu;     // mode 0
    float* out;          // mode 0: G (S, D); mode 1: dL (D, D)
    float* ws;           // mode 0: partial accumulators [unit][n][128]
};

// unit -> (row block, chunk) for the triangle with q column blocks per chunk: row blocks g q .. g q + q - 1 have g + 1 units each
__host__ __device__ inline void tri_unit(int u, int q, int& rb, int& chunk)
{
    int g = 0;
    while (q * (g + 1) * (g + 2) / 2 <= u) ++g;
    const int r = u - q * g * (g + 1) / 2;
    rb = g * q + r / (g + 1);
    chunk = r % (g + 1);
}
__host__ __device__ inline int tri_unit_base(int rb, int q)
{
    const int g = rb / q;
    return q * g * (g + 1) / 2 + (rb - g * q) * (g + 1);
}

__global__ void __launch_bounds__(DG_THREADS, 1)
dense_gemm_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, const DenseGemmArgs p, int stages)
{
    extern __shared__ unsigned char dsm_raw[];
    __shared__ uint64_t full_bar[3], split_bar[3], empty_bar[3], acc_bar;
    unsigned char* dsm = dsm_raw + ((1024u - (smem_u32(dsm_raw) & 1023u)) & 1023u);   // 128-byte swizzle atoms: 1024-byte aligned tiles
    __shared__ uint32_t tmem_base_smem;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int N = p.n;
    const uint32_t tile_b = uint32_t(N) * DG_BK * 4;
    const uint32_t stage_bytes = 2 * DG_TILE_A + 2 * tile_b;   // A raw, A lo, B raw, B lo
    uint32_t tm_cols = 32;
    while (tm_cols < uint32_t(N)) tm_cols <<= 1;

    // ---- what this CTA computes
    int row_blk, col_blk = 0, kb0, nkb, chunk = 0;
    if (p.mode == 0) {
        tri_unit(blockIdx.x, p.q, row_blk, chunk);
        kb0 = chunk * p.q * (DG_BM / DG_BK);
        const int kend = min((chunk + 1) * p.q, row_blk + 1) * (DG_BM / DG_BK);
        nkb = kend - kb0;
    } else {
        int ti = 0;
        while ((ti + 1) * (ti + 2) / 2 <= int(blockIdx.x)) ++ti;
        row_blk = ti;
        col_blk = int(blockIdx.x) - ti * (ti + 1) / 2;
        kb0 = 0;
        nkb = p.k_blocks_total;
    }
    const int row0 = row_blk * DG_BM;

    if (threadIdx.x == 0) {
        for (int i = 0; i < stages; ++i) {
            mbar_init(&full_bar[i], 1);
            mbar_init(&split_bar[i], 128);
            mbar_init(&empty_bar[i], 1);
        }
        mbar_init(&acc_bar, 1);
        mbar_fence_init();
    }
    if (warp == 1) tm_alloc(&tmem_base_smem, tm_cols);
    tm_fence_before();
    __syncthreads();
    tm_fence_after();
    const uint32_t tmem_acc = tmem_base_smem;

    if (warp == 0) {
        // ------------------------------------------------------------------ TMA producer
        if (lane == 0) {
            for (int i = 0; i < nkb; ++i) {
                const int st = i % stages;
                if (i >= stages) mbar_wait(&empty_bar[st], ((i / stages) & 1) ^ 1);
                unsigned char* stage = dsm + size_t(st) * stage_bytes;
                mbar_arrive_expect_tx(&full_bar[st], DG_TILE_A + tile_b);
                const int kcol = (kb0 + i) * DG_BK;
                tma_load_2d(stage, &map_a, kcol, row0, &full_bar[st]);
                tma_load_2d(stage + 2 * DG_TILE_A, &map_b, kcol, p.mode == 0 ? 0 : col_blk * DG_BM, &full_bar[st]);
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------------ MMA issuer (one thread)
        if (lane == 0) {
            const uint32_t idesc = umma_idesc_tf32(DG_BM, N);
            for (int i = 0; i < nkb; ++i) {
                const int st = i % stages;
                mbar_wait(&split_bar[st], (i / stages) & 1);
                tm_fence_after();
                const uint32_t a_hi = smem_u32(dsm + size_t(st) * stage_bytes), a_lo = a_hi + DG_TILE_A;
                const uint32_t b_hi = a_hi + 2 * DG_TILE_A, b_lo = b_hi + tile_b;
#pragma unroll
                for (int ks = 0; ks < DG_BK / 8; ++ks) {   // K = 8 tf32 = 32 bytes inside the 128-byte swizzle row
                    const uint64_t dah = umma_desc_sw128(a_hi + ks * 32), dal = umma_desc_sw128(a_lo + ks * 32);
                    const uint64_t dbh = umma_desc_sw128(b_hi + ks * 32), dbl = umma_desc_sw128(b_lo + ks * 32);
                    umma_tf32(tmem_acc, dah, dbh, idesc, (i | ks) != 0);
                    umma_tf32(tmem_acc, dah, dbl, idesc, 1);
                    umma_tf32(tmem_acc, dal, dbh, idesc, 1);
                }
                umma_commit(&empty_bar[st]);   // arrives when the MMAs that read this stage are done
            }
            umma_commit(&acc_bar);
        }
    } else {
        // ------------------------------------------------------------------ operand split, then epilogue
        const int t = threadIdx.x - 64;   // 0..127
        for (int i = 0; i < nkb; ++i) {
            const int st = i % stages;
            mbar_wait(&full_bar[st], (i / stages) & 1);
            unsigned char* stage = dsm + size_t(st) * stage_bytes;
            const int kcol = (kb0 + i) * DG_BK;
            // mode 0: blocks that reach past the first row of this row block straddle the diagonal of L
            const bool diag = p.mode == 0 && kcol + DG_BK > row0 + 1;
            for (int c = t; c < DG_BM * 8; c += 128) {   // A: 16-byte chunks; physical chunk pc of row r holds columns 4 (pc ^ (r & 7)) ..
                float4 x = *reinterpret_cast<const float4*>(stage + c * 16);
                if (diag) {
                    const int r = c >> 3, col = kcol + 4 * ((c & 7) ^ (r & 7)), i_row = row0 + r;
                    if (col + 0 > i_row) x.x = 0.f;
                    if (col + 1 > i_row) x.y = 0.f;
                    if (col + 2 > i_row) x.z = 0.f;
                    if (col + 3 > i_row) x.w = 0.f;
                    *reinterpret_cast<float4*>(stage + c * 16) = x;   // the masked raw tile is the hi operand
                }
                float4 lo;
                lo.x = x.x - __uint_as_float(__float_as_uint(x.x) & 0xFFFFE000u);
                lo.y = x.y - __uint_as_float(__float_as_uint(x.y) & 0xFFFFE000u);
                lo.z = x.z - __uint_as_float(__float_as_uint(x.z) & 0xFFFFE000u);
                lo.w = x.w - __uint_as_float(__float_as_uint(x.w) & 0xFFFFE000u);
                *reinterpret_cast<float4*>(stage + DG_TILE_A + c * 16) = lo;
            }
            unsigned char* braw = stage + 2 * DG_TILE_A;
            for (int c = t; c < N * 8; c += 128) {
                const float4 x = *reinterpret_cast<const float4*>(braw + c * 16);
                float4 lo;
                lo.x = x.x - __uint_as_float(__float_as_uint(x.x) & 0xFFFFE000u);
                lo.y = x.y - __uint_as_float(__float_as_uint(x.y) & 0xFFFFE000u);
                lo.z = x.z - __uint_as_float(__float_as_uint(x.z) & 0xFFFFE000u);
                lo.w = x.w - __uint_as_float(__float_as_uint(x.w) & 0xFFFFE000u);
                *reinterpret_cast<float4*>(braw + tile_b + c * 16) = lo;
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> visible to the MMA
            mbar_arrive(&split_bar[st]);
        }
        // epilogue: this warp reads its TMEM lane quadrant (warp % 4): lane = row m of the unit
        mbar_wait(&acc_bar, 0);
        tm_fence_after();
        const int quad = warp & 3;
        const int m = 32 * quad + lane;
        const uint32_t taddr = tmem_acc + (uint32_t(32 * quad) << 16);
        if (p.mode == 0) {
            const int i_row = row0 + m;
            const bool single = row_blk < p.q;   // one unit covers the whole row block: write G directly
            const float mu = single ? p.mu[i_row] : 0.f;
            float* wsu = p.ws + (size_t(blockIdx.x) * N) * DG_BM + m;
            for (int c = 0; c < N; c += 16) {
                float v[16];
                tm_ld16(v, taddr + c);
                tm_wait_ld();
#pragma unroll
                for (int s = 0; s < 16; ++s) {
                    if (single) {
                        if (c + s < p.S) p.out[size_t(c + s) * p.D + i_row] = v[s] + mu;
                    } else {
                        wsu[size_t(c + s) * DG_BM] = v[s];
                    }
                }
            }
        } else {
            const int i_row = row0 + m;
            float* orow = p.out + size_t(i_row) * p.D + size_t(col_blk) * DG_BM;
            const bool diag_tile = col_blk == row_blk;
            for (int c = 0; c < DG_BM; c += 16) {
                float v[16];
                tm_ld16(v, taddr + c);
                tm_wait_ld();
                if (diag_tile) {
#pragma unroll
                    for (int s = 0; s < 16; ++s)
                        if (col_blk * DG_BM + c + s > i_row) v[s] = 0.f;
                }
#pragma unroll
                for (int s = 0; s < 16; s += 4) *reinterpret_cast<float4*>(orow + c + s) = make_float4(v[s], v[s + 1], v[s + 2], v[s + 3]);
            }
        }
    }
    tm_fence_before();
    __syncthreads();
    if (warp == 1) tm_dealloc(tmem_acc, tm_cols);
}

// G[s, i] = mu[i] + sum over the row block's units (fixed order) of the partial accumulators; row blocks >= q only
__global__ void __launch_bounds__(128)
dense_reparam_reduce_kernel(const float* __restrict__ ws, const float* __restrict__ mu, float* __restrict__ g, int S, int D, int n, int q)
{
    const int rb = blockIdx.x + q, s = blockIdx.y, m = threadIdx.x;
    if (s >= S) return;
    const int base = tri_unit_base(rb, q), cnt = rb / q + 1;
    float acc = 0.f;
    for (int c = 0; c < cnt; ++c) acc += ws[(size_t(base + c) * n + s) * DG_BM + m];
    const int i = rb * DG_BM + m;
    g[size_t(s) * D + i] = acc + mu[i];
}

// ---- tensor maps ---------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn()
{
    static EncodeTiledFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess || qres != cudaDriverEntryPointSuccess)
            p = nullptr;
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    return fn;
}
// row-major fp32 matrix (rows x cols, leading dimension ld floats), boxes of 32 columns x box_rows rows, 128-byte swizzle,
// out-of-bounds elements read as zero
static int make_map(CUtensorMap* map, const float* base, int64_t rows, int64_t cols, int64_t ld, int box_rows)
{
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn) return fail(WHVI_E_MODE, "dense GEMM: cuTensorMapEncodeTiled is not available from this driver");
    const cuuint64_t dims[2] = {cuuint64_t(cols), cuuint64_t(rows)};
    const cuuint64_t strides[1] = {cuuint64_t(ld) * sizeof(float)};
    const cuuint32_t box[2] = {DG_BK, cuuint32_t(box_rows)};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(WHVI_E_SHAPE, "dense GEMM: cuTensorMapEncodeTiled failed (%d)", int(r));
    return WHVI_OK;
}

static int launch_dense_gemm(const CUtensorMap& ma, const CUtensorMap& mb, const DenseGemmArgs& a, int64_t units, cudaStream_t stream)
{
    static unsigned char smem_ok[64] = {};
    const int stages = a.n <= 128 ? 3 : 2;
    const size_t smem = size_t(stages) * (2 * DG_TILE_A + 2 * size_t(a.n) * DG_BK * 4) + 1024;
    if (int rc = ensure_smem(dense_gemm_kernel, 200 * 1024, smem_ok)) return rc;   // opt in once for the largest configuration
    dense_gemm_kernel<<<static_cast<unsigned>(units), DG_THREADS, smem, stream>>>(ma, mb, a, stages);
    return check_launch("dense_gemm_kernel");
}

// q: column blocks per unit such that the triangle splits into about 3 waves of units at most, at least 4
static int dense_q(int64_t D)
{
    const int64_t RB = D / DG_BM;
    int q = 4;
    while (true) {
        int64_t units = 0;
        for (int64_t rb = 0; rb < RB; ++rb) units += rb / q + 1;
        if (units <= 148 * 3 || q >= RB) break;
        q *= 2;
    }
    return q;
}

size_t reparam_dense_workspace_bytes(int64_t S, int64_t D)
{
    const int q = dense_q(D);
    const int64_t RB = D / DG_BM;
    int64_t units = 0;
    for (int64_t rb = 0; rb < RB; ++rb) units += rb / q + 1;
    const int64_t ns = S < 256 ? S : 256;
    const int64_t NP = (ns + 15) / 16 * 16;
    return sizeof(float) * size_t(units) * NP * DG_BM;
}

int launch_reparam_dense(const float* mu, const float* L, const float* eps, float* g, int64_t S, int64_t D, float* ws, size_t ws_bytes,
                         cudaStream_t stream)
{
    if (D % DG_BM != 0) return fail(WHVI_E_SHAPE, "reparam(dense): D = %lld must be a multiple of 128", (long long)D);
    if (ws == nullptr || ws_bytes < reparam_dense_workspace_bytes(S, D))
        return fail(WHVI_E_WORKSPACE, "reparam(dense): workspace of %zu bytes needed, %zu given", reparam_dense_workspace_bytes(S, D), ws_bytes);
    const int q = dense_q(D);
    const int64_t RB = D / DG_BM;
    int64_t units = 0;
    for (int64_t rb = 0; rb < RB; ++rb) units += rb / q + 1;
    CUtensorMap ma, mb;
    if (int rc = make_map(&ma, L, D, D, D, DG_BM)) return rc;
    for (int64_t s0 = 0; s0 < S; s0 += 256) {   // sample blocks of up to 256 (the MMA's N)
        const int ns = static_cast<int>(S - s0 < 256 ? S - s0 : 256);
        const int NP = (ns + 15) / 16 * 16;
        if (int rc = make_map(&mb, eps + s0 * D, ns, D, D, NP)) return rc;
        DenseGemmArgs a{0, NP, q, 0, static_cast<int>(D), ns, mu, g + s0 * D, ws};
        if (int rc = launch_dense_gemm(ma, mb, a, units, stream)) return rc;
        if (RB > q) {
            dim3 grid(static_cast<unsigned>(RB - q), static_cast<unsigned>(ns));
            dense_reparam_reduce_kernel<<<grid, 128, 0, stream>>>(ws, mu, g + s0 * D, ns, static_cast<int>(D), NP, q);
            if (int rc = check_launch("dense_reparam_reduce_kernel")) return rc;
        }
    }
    return WHVI_OK;
}

// dL = tril(dgT ET^T): dgT, ET are (D, Sp) row-major (the caller's transposes of dG and E, zero-padded to Sp % 32 == 0)
int launch_reparam_dense_bwd(const float* dgT, const float* eT, float* dL, int64_t Sp, int64_t D, cudaStream_t stream)
{
    if (D % DG_BM != 0 || Sp % DG_BK != 0 || Sp <= 0) return fail(WHVI_E_SHAPE, "reparam_bwd(dense): D %% 128 == 0 and padded S %% 32 == 0 required");
    CUtensorMap ma, mb;
    if (int rc = make_map(&ma, dgT, D, Sp, Sp, DG_BM)) return rc;
    if (int rc = make_map(&mb, eT, D, Sp, Sp, DG_BM)) return rc;
    const int64_t RB = D / DG_BM;
    DenseGemmArgs a{1, DG_BM, 0, static_cast<int>(Sp / DG_BK), static_cast<int>(D), 0, nullptr, dL, nullptr};
    return launch_dense_gemm(ma, mb, a, RB * (RB + 1) / 2, stream);
}

// ---- kernel (5), dense: KL( N(mu, L L^T) || N(0, lambda I) ) and its gradients -----------------------------------------
// one CTA per row of L: row sums of squares of the lower triangle (dL = grad_scale * L / lambda written on the way, zero
// above the diagonal), then a fixed-order fp64 combination by a second tiny kernel.
__global__ void __launch_bounds__(256)
kl_dense_rows_kernel(const float* __restrict__ L, float lambda_, int D, float* __restrict__ dL, float grad_scale, double* __restrict__ row_sq)
{
    __shared__ double red[8];
    const int i = blockIdx.x;
    const float inv_l = 1.f / lambda_;
    double acc = 0.0;
    for (int j = threadIdx.x; j < D; j += blockDim.x) {
        const float v = j <= i ? L[size_t(i) * D + j] : 0.f;
        acc += double(v) * double(v);
        if (dL) {
            float gr = grad_scale * v * inv_l;
            if (j == i) gr -= grad_scale / v;
            dL[size_t(i) * D + j] = gr;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double tot = 0.0;
        for (int w = 0; w < 8; ++w) tot += red[w];
        row_sq[i] = tot;
    }
}
__global__ void __launch_bounds__(1024)
kl_dense_final_kernel(const float* __restrict__ mu, const float* __restrict__ L, float lambda_, int D, const double* __restrict__ row_sq,
                      float* __restrict__ out, float* __restrict__ dmu, float grad_scale)
{
    __shared__ double red[3][32];
    double s_sq = 0.0, s_log = 0.0, s_mu = 0.0;
    const float inv_l = 1.f / lambda_;
    for (int i = threadIdx.x; i < D; i += blockDim.x) {
        s_sq += row_sq[i];
        s_log += log(double(L[size_t(i) * D + i]));
        const float m = mu[i];
        s_mu += double(m) * double(m);
        if (dmu) dmu[i] = grad_scale * m * inv_l;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s_sq += __shfl_xor_sync(0xffffffffu, s_sq, o);
        s_log += __shfl_xor_sync(0xffffffffu, s_log, o);
        s_mu += __shfl_xor_sync(0xffffffffu, s_mu, o);
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) red[0][warp] = s_sq, red[1][warp] = s_log, red[2][warp] = s_mu;
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0.0, b = 0.0, c = 0.0;
        for (int w = 0; w < int(blockDim.x >> 5); ++w) a += red[0][w], b += red[1][w], c += red[2][w];
        const double d = double(D), lam = double(lambda_);
        out[0] = static_cast<float>(0.5 * (d * log(lam) - 2.0 * b - d + a / lam + c / lam));
    }
}

int launch_kl_dense(const float* mu, const float* L, float lambda_, int64_t D, float* out, float* dmu, float* dL, float grad_scale,
                    double* row_sq /* D doubles of workspace */, cudaStream_t stream)
{
    kl_dense_rows_kernel<<<static_cast<unsigned>(D), 256, 0, stream>>>(L, lambda_, static_cast<int>(D), dL, grad_scale, row_sq);
    if (int rc = check_launch("kl_dense_rows_kernel")) return rc;
    int threads = 32;
    while (threads < D && threads < 1024) threads <<= 1;
    kl_dense_final_kernel<<<1, threads, 0, stream>>>(mu, L, lambda_, static_cast<int>(D), row_sq, out, dmu, grad_scale);
    return check_launch("kl_dense_final_kernel");
}

// ---- grouped forms: G blocks (the square blocks of a Stacked layer), block k's mu at + k * mu_stride floats and its L at
// + k * L_stride; eps, g, dg: (G, S, D); dmu (G, D) and dL (G, D, D) are written densely.
//
// D <= 64: one CUDA-core kernel per direction for all blocks.  L_k (at most 64 x 64) sits in shared memory with a padded row
// (no bank conflicts on the column walk); every output is one fp32 chain in a fixed order (j ascending forward, s ascending
// backward), so the results are bit-reproducible.  The tcgen05 GEMM above cannot take these widths (its tile is 128 rows).
constexpr int RDS_THREADS = 256;
constexpr int RDS_MAX_D = 64;

// grid (ceil(S / ST), G), ST = samples per CTA
__global__ void __launch_bounds__(RDS_THREADS)
reparam_dense_small_kernel(const float* __restrict__ mu, int64_t mu_stride, const float* __restrict__ L, int64_t L_stride,
                           const float* __restrict__ eps, float* __restrict__ g, int S, int D, int ST)
{
    __shared__ float Ls[RDS_MAX_D * (RDS_MAX_D + 1)];
    __shared__ float es[RDS_THREADS * 16];   // ST * D <= 4096
    const int k = blockIdx.y, s0 = blockIdx.x * ST;
    const int ns = min(ST, S - s0);
    const float* Lk = L + size_t(k) * L_stride;
    const float* muk = mu + size_t(k) * mu_stride;
    for (int e = threadIdx.x; e < D * D; e += RDS_THREADS) {
        const int i = e / D, j = e - i * D;
        Ls[i * (D + 1) + j] = j <= i ? Lk[e] : 0.f;
    }
    const float* ek = eps + (size_t(k) * S + s0) * D;
    for (int e = threadIdx.x; e < ns * D; e += RDS_THREADS) es[e] = ek[e];
    __syncthreads();
    float* gk = g + (size_t(k) * S + s0) * D;
    for (int e = threadIdx.x; e < ns * D; e += RDS_THREADS) {
        const int s = e / D, i = e - s * D;
        const float* lr = Ls + i * (D + 1);
        const float* er = es + s * D;
        float acc = 0.f;
        for (int j = 0; j <= i; ++j) acc = fmaf(lr[j], er[j], acc);
        gk[e] = muk[i] + acc;
    }
}

// dL_k[i, j] = sum_s dg[k, s, i] eps[k, s, j] (j <= i, 0 above), dmu_k[i] = sum_s dg[k, s, i].  Thread e of the block's
// D * D + D outputs: e < D * D is entry (e / D, e % D) of dL_k, the rest dmu_k.  grid (ceil((D * D + D) / 256), G); the samples
// pass through shared memory in tiles of RDS_TILE_S rows.
constexpr int RDS_TILE_S = 32;
__global__ void __launch_bounds__(RDS_THREADS)
reparam_dense_small_bwd_kernel(const float* __restrict__ eps, const float* __restrict__ dg, float* __restrict__ dmu, float* __restrict__ dL,
                               int S, int D)
{
    __shared__ float dgs[RDS_TILE_S * RDS_MAX_D], es[RDS_TILE_S * RDS_MAX_D];
    const int k = blockIdx.y;
    const int e = blockIdx.x * RDS_THREADS + threadIdx.x;
    const int DD = D * D;
    int i = 0, j = -1;   // j = -1: dmu entry
    bool active = false;
    if (e < DD) {
        i = e / D, j = e - (e / D) * D;
        active = j <= i;
    } else if (e < DD + D) {
        i = e - DD;
        active = true;
    }
    const float* dgk = dg + size_t(k) * S * D;
    const float* ek = eps + size_t(k) * S * D;
    float acc = 0.f;
    for (int s0 = 0; s0 < S; s0 += RDS_TILE_S) {
        const int ns = min(RDS_TILE_S, S - s0);
        __syncthreads();
        for (int t = threadIdx.x; t < ns * D; t += RDS_THREADS) {
            dgs[t] = dgk[size_t(s0) * D + t];
            es[t] = ek[size_t(s0) * D + t];
        }
        __syncthreads();
        if (active) {
            if (j >= 0)
                for (int s = 0; s < ns; ++s) acc = fmaf(dgs[s * D + i], es[s * D + j], acc);
            else
                for (int s = 0; s < ns; ++s) acc += dgs[s * D + i];
        }
    }
    if (e < DD)
        dL[size_t(k) * DD + e] = acc;   // 0 above the diagonal
    else if (e < DD + D)
        dmu[size_t(k) * D + i] = acc;
}

// D >= 128: the K-major operands of the dL GEMM for block k, dgT / eT (D, Sp) = the transposes of dg / eps (S, D), zero past
// S.  32 x 32 tiles through shared memory; grid (Sp / 32, D / 32).
__global__ void __launch_bounds__(256)
dense_transpose_pad_kernel(const float* __restrict__ dg, const float* __restrict__ eps, float* __restrict__ dgT, float* __restrict__ eT,
                           int S, int D, int Sp)
{
    __shared__ float ta[32][33], tb[32][33];
    const int s0 = blockIdx.x * 32, i0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    for (int r = ty; r < 32; r += 8) {
        const int s = s0 + r;
        ta[r][tx] = s < S ? dg[size_t(s) * D + i0 + tx] : 0.f;
        tb[r][tx] = s < S ? eps[size_t(s) * D + i0 + tx] : 0.f;
    }
    __syncthreads();
    for (int r = ty; r < 32; r += 8) {
        dgT[size_t(i0 + r) * Sp + s0 + tx] = ta[tx][r];
        eT[size_t(i0 + r) * Sp + s0 + tx] = tb[tx][r];
    }
}

// dmu[k, i] = sum_s dg[k, s, i], samples ascending
__global__ void __launch_bounds__(256)
dense_colsum_kernel(const float* __restrict__ dg, float* __restrict__ dmu, int S, int D)
{
    const int k = blockIdx.y, i = blockIdx.x * 256 + threadIdx.x;
    if (i >= D) return;
    const float* p = dg + size_t(k) * S * D + i;
    float acc = 0.f;
    for (int s = 0; s < S; ++s) acc += p[size_t(s) * D];
    dmu[size_t(k) * D + i] = acc;
}

static int64_t round_up(int64_t v, int64_t m) { return (v + m - 1) / m * m; }

size_t reparam_dense_grouped_workspace_bytes(int64_t S, int64_t D)
{
    if (D < DG_BM) return 0;
    const size_t fwd = reparam_dense_workspace_bytes(S, D);
    const size_t bwd = sizeof(float) * 2 * size_t(D) * size_t(round_up(S < 1 ? 1 : S, DG_BK));
    return fwd > bwd ? fwd : bwd;
}

int launch_reparam_dense_grouped(const float* mu, int64_t mu_stride, const float* L, int64_t L_stride, const float* eps, float* g, int64_t S,
                                 int64_t D, int64_t G, float* ws, size_t ws_bytes, cudaStream_t stream)
{
    if (D <= RDS_MAX_D) {
        const int ST = static_cast<int>(D >= 16 ? 4096 / D : 256);
        const dim3 grid(static_cast<unsigned>((S + ST - 1) / ST), static_cast<unsigned>(G));
        reparam_dense_small_kernel<<<grid, RDS_THREADS, 0, stream>>>(mu, mu_stride, L, L_stride, eps, g, static_cast<int>(S), static_cast<int>(D), ST);
        return check_launch("reparam_dense_small_kernel");
    }
    for (int64_t k = 0; k < G; ++k)   // one tcgen05 reparameterisation per block (G = ceil(n_out / D) is small)
        if (int rc = launch_reparam_dense(mu + k * mu_stride, L + k * L_stride, eps + k * S * D, g + k * S * D, S, D, ws, ws_bytes, stream))
            return rc;
    return WHVI_OK;
}

int launch_reparam_dense_grouped_bwd(const float* eps, const float* dg, float* dmu, float* dL, int64_t S, int64_t D, int64_t G, float* ws,
                                     size_t ws_bytes, cudaStream_t stream)
{
    if (D <= RDS_MAX_D) {
        const dim3 grid(static_cast<unsigned>((D * D + D + RDS_THREADS - 1) / RDS_THREADS), static_cast<unsigned>(G));
        reparam_dense_small_bwd_kernel<<<grid, RDS_THREADS, 0, stream>>>(eps, dg, dmu, dL, static_cast<int>(S), static_cast<int>(D));
        return check_launch("reparam_dense_small_bwd_kernel");
    }
    if (ws == nullptr || ws_bytes < reparam_dense_grouped_workspace_bytes(S, D))
        return fail(WHVI_E_WORKSPACE, "reparam_bwd(dense, grouped): workspace of %zu bytes needed, %zu given",
                    reparam_dense_grouped_workspace_bytes(S, D), ws_bytes);
    const int64_t Sp = round_up(S, DG_BK);
    float* dgT = ws;
    float* eT = ws + D * Sp;
    // the GEMM writes the tiles on and below the diagonal only
    if (cudaMemsetAsync(dL, 0, sizeof(float) * size_t(G) * D * D, stream) != cudaSuccess) return check_launch("reparam_bwd(dense): memset");
    for (int64_t k = 0; k < G; ++k) {
        const dim3 tgrid(static_cast<unsigned>(Sp / 32), static_cast<unsigned>(D / 32));
        dense_transpose_pad_kernel<<<tgrid, 256, 0, stream>>>(dg + k * S * D, eps + k * S * D, dgT, eT, static_cast<int>(S), static_cast<int>(D),
                                                              static_cast<int>(Sp));
        if (int rc = check_launch("dense_transpose_pad_kernel")) return rc;
        if (int rc = launch_reparam_dense_bwd(dgT, eT, dL + k * D * D, Sp, D, stream)) return rc;
    }
    const dim3 cgrid(static_cast<unsigned>((D + 255) / 256), static_cast<unsigned>(G));
    dense_colsum_kernel<<<cgrid, 256, 0, stream>>>(dg, dmu, static_cast<int>(S), static_cast<int>(D));
    return check_launch("dense_colsum_kernel");
}

// Sum over G blocks of the dense KL: the row kernel with a block axis (grid (D, G)), then one CTA that adds the rows' squares,
// the log-diagonals and |mu|^2 in a fixed order (blocks ascending inside every thread's strided walk).
__global__ void __launch_bounds__(256)
kl_dense_grouped_rows_kernel(const float* __restrict__ L, int64_t L_stride, float lambda_, int D, float* __restrict__ dL, float grad_scale,
                             double* __restrict__ row_sq)
{
    __shared__ double red[8];
    const int i = blockIdx.x, k = blockIdx.y;
    const float* Lk = L + size_t(k) * L_stride;
    float* dLk = dL ? dL + size_t(k) * D * D : nullptr;
    const float inv_l = 1.f / lambda_;
    double acc = 0.0;
    for (int j = threadIdx.x; j < D; j += blockDim.x) {
        const float v = j <= i ? Lk[size_t(i) * D + j] : 0.f;
        acc += double(v) * double(v);
        if (dLk) {
            float gr = grad_scale * v * inv_l;
            if (j == i) gr -= grad_scale / v;
            dLk[size_t(i) * D + j] = gr;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double tot = 0.0;
        for (int w = 0; w < int(blockDim.x >> 5); ++w) tot += red[w];
        row_sq[size_t(k) * D + i] = tot;
    }
}
__global__ void __launch_bounds__(1024)
kl_dense_grouped_final_kernel(const float* __restrict__ mu, int64_t mu_stride, const float* __restrict__ L, int64_t L_stride, float lambda_,
                              int D, int G, const double* __restrict__ row_sq, float* __restrict__ out, float* __restrict__ dmu, float grad_scale)
{
    __shared__ double red[3][32];
    double s_sq = 0.0, s_log = 0.0, s_mu = 0.0;
    const float inv_l = 1.f / lambda_;
    for (int k = 0; k < G; ++k) {
        const float* Lk = L + size_t(k) * L_stride;
        const float* muk = mu + size_t(k) * mu_stride;
        for (int i = threadIdx.x; i < D; i += blockDim.x) {
            s_sq += row_sq[size_t(k) * D + i];
            s_log += log(double(Lk[size_t(i) * D + i]));
            const float m = muk[i];
            s_mu += double(m) * double(m);
            if (dmu) dmu[size_t(k) * D + i] = grad_scale * m * inv_l;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s_sq += __shfl_xor_sync(0xffffffffu, s_sq, o);
        s_log += __shfl_xor_sync(0xffffffffu, s_log, o);
        s_mu += __shfl_xor_sync(0xffffffffu, s_mu, o);
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) red[0][warp] = s_sq, red[1][warp] = s_log, red[2][warp] = s_mu;
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0.0, b = 0.0, c = 0.0;
        for (int w = 0; w < int(blockDim.x >> 5); ++w) a += red[0][w], b += red[1][w], c += red[2][w];
        const double n = double(D) * double(G), lam = double(lambda_);
        out[0] = static_cast<float>(0.5 * (n * log(lam) - 2.0 * b - n + a / lam + c / lam));
    }
}

int launch_kl_dense_grouped(const float* mu, int64_t mu_stride, const float* L, int64_t L_stride, float lambda_, int64_t D, int64_t G, float* out,
                            float* dmu, float* dL, float grad_scale, double* row_sq /* G * D doubles */, cudaStream_t stream)
{
    const int threads = D >= 256 ? 256 : 32;
    kl_dense_grouped_rows_kernel<<<dim3(static_cast<unsigned>(D), static_cast<unsigned>(G)), threads, 0, stream>>>(
        L, L_stride, lambda_, static_cast<int>(D), dL, grad_scale, row_sq);
    if (int rc = check_launch("kl_dense_grouped_rows_kernel")) return rc;
    int ft = 32;
    while (ft < D && ft < 1024) ft <<= 1;
    kl_dense_grouped_final_kernel<<<1, ft, 0, stream>>>(mu, mu_stride, L, L_stride, lambda_, static_cast<int>(D), static_cast<int>(G), row_sq, out,
                                                        dmu, grad_scale);
    return check_launch("kl_dense_grouped_final_kernel");
}

}  // namespace whvi
