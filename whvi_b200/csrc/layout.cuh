// Compile-time data layouts ("views") for the register/shared-memory FWHT engine.
//
// A tile is N = 2^n consecutive floats (one row of length D = N, or N/D whole rows when
// D < N).  It is processed by T = 2^t threads holding E = 2^c floats each (n = t + c).
// A *view* says which logical index bit every register-index bit and every thread-id
// bit stands for.  A butterfly on logical bit b is register-local in any view where b
// is a register bit, so a transform is a sequence of views ("rounds") whose register
// bits together cover the transform bits, with a shared-memory transposition between
// consecutive views.
//
// Constraints baked into the three canonical views (checked by tools/sim_layout.cpp):
//  * FIRST / LAST: register bits 0,1 = logical bits 0,1 (one float4) and lanes =
//    logical bits 2..6, so global accesses are 128-bit and a warp touches 512
//    contiguous bytes per instruction.
//  * The physical shared-memory layout of a transposition is defined by the READER
//    view: thread tid' owns E consecutive words, read as float4 slots XOR-swizzled by
//    tid' so that each quarter-warp covers all eight 16-byte bank groups.
//  * The WRITER's lanes map one-to-one onto the 32 banks (scalar STS), which holds
//    because its five lane bits are the reader's register bits 0..4.
//
// Everything here is constexpr and host/device so the same code drives the kernels and
// the host simulator.
#pragma once
#include <cstdint>

#if defined(__CUDACC__)
#define WHVI_HD __host__ __device__ __forceinline__
#else
#define WHVI_HD inline
#endif

// WHVI_PADDED=1 (defined by layer_bwd.cu and layer_loss.cu before they include this file):
// the reader-owned transposition layout without the XOR swizzle -- thread tid' owns E + 4 words at
// tid' * (E + 4), register r at word r.  Conflict-free on both sides like the swizzle
// (tools/sim_layout.cpp proves it for every transposition in use) and every address is a thread
// base plus a compile-time constant (no LOP3 per access), at 12.5% more scratch.  Measured ~4% faster
// in the backward and no faster in the two-view forward (profiles/r02_ab_padbwd.txt), so the other
// translation units keep the swizzled layout.
#ifndef WHVI_PADDED
#define WHVI_PADDED 0
#endif

namespace whvi {

constexpr int kMaxBits = 16;

// words of one transposition buffer (or MID-order g table) of a 2^n tile, 2^c floats per thread
constexpr uint32_t scratch_words(int n, int c) { return (1u << n) + (WHVI_PADDED ? (4u << (n - c)) : 0u); }

struct View {
    int n;               // log2(tile elements)
    int c;               // log2(elements per thread)
    int bit[kMaxBits];   // bit[p], p < c: register bit p; p >= c: thread-id bit p - c
};

constexpr bool view_has(const View& v, int upto, int b)
{
    for (int p = 0; p < upto; ++p)
        if (v.bit[p] == b) return true;
    return false;
}

// Append every logical bit not yet present, ascending (fills the thread-id bits).
constexpr View view_fill(View v, int used)
{
    for (int b = 0; b < v.n; ++b)
        if (!view_has(v, used, b)) v.bit[used++] = b;
    return v;
}

// FIRST view: registers = {0,1} + the top c-2 bits; lanes = 2..6.
constexpr View view_first(int n, int c)
{
    View v{n, c, {}};
    v.bit[0] = 0;
    v.bit[1] = 1;
    for (int i = 0; i < c - 2; ++i) v.bit[2 + i] = n - (c - 2) + i;
    for (int i = 0; i < 5; ++i) v.bit[c + i] = 2 + i;
    return view_fill(v, c + 5);
}

// MID view registers: 2..6 plus (c-5) more bits starting at 7.
constexpr int mid_reg_bit(int c, int p) { return p < 5 ? 2 + p : 7 + (p - 5); }

// LAST view: registers = {0,1}, then the first three bits >= 7 that are not MID register
// bits (they double as MID's lanes), then further bits (fillers if n is exhausted);
// lanes = 2..6.
constexpr View view_last(int n, int c)
{
    View v{n, c, {}};
    v.bit[0] = 0;
    v.bit[1] = 1;
    int next = 7 + (c - 5);
    for (int p = 2; p < c; ++p) {
        if (next < n) {
            v.bit[p] = next++;
        } else {  // out of fresh bits: reuse a MID register bit >= 7 as a filler
            int f = 7;
            while (view_has(v, p, f)) ++f;
            v.bit[p] = f;
        }
    }
    for (int i = 0; i < 5; ++i) v.bit[c + i] = 2 + i;
    return view_fill(v, c + 5);
}

// MID view: registers = 2..6 (+ bits 7.. for c > 5); lanes = {0,1} + register bits 2..4 of
// the view it is transposed INTO next (`toward`): LAST on the way forward (MID), FIRST on
// the way back (MID2).  Remaining thread bits ascending.
constexpr View view_mid_toward(int n, int c, const View& toward)
{
    View v{n, c, {}};
    for (int p = 0; p < c; ++p) v.bit[p] = mid_reg_bit(c, p);
    v.bit[c + 0] = 0;
    v.bit[c + 1] = 1;
    v.bit[c + 2] = toward.bit[2];
    v.bit[c + 3] = toward.bit[3];
    v.bit[c + 4] = toward.bit[4];
    return view_fill(v, c + 5);
}
constexpr View view_mid(int n, int c) { return view_mid_toward(n, c, view_last(n, c)); }

// MID2 needs FIRST's register bits 2..4 as lanes; when one of them is a MID register bit
// (c == 6, n == 11: bit 7) fall back to MID (that configuration is 2-round anyway and
// MID -> FIRST is conflict-free there).
constexpr View view_mid2(int n, int c)
{
    const View f = view_first(n, c);
    for (int p = 2; p < 5; ++p)
        for (int q = 0; q < c; ++q)
            if (f.bit[p] == mid_reg_bit(c, q)) return view_mid(n, c);
    return view_mid_toward(n, c, f);
}

// position of logical bit b inside the view (index into View::bit)
constexpr int view_pos(const View& v, int b)
{
    for (int p = 0; p < v.n; ++p)
        if (v.bit[p] == b) return p;
    return -1;
}

// logical index contributed by a register index / a thread id
constexpr uint32_t view_reg_logical(const View& v, uint32_t reg)
{
    uint32_t idx = 0;
    for (int p = 0; p < v.c; ++p) idx |= ((reg >> p) & 1u) << v.bit[p];
    return idx;
}
WHVI_HD uint32_t view_tid_logical(const View& v, uint32_t tid)
{
    uint32_t idx = 0;
    for (int p = v.c; p < v.n; ++p) idx |= ((tid >> (p - v.c)) & 1u) << v.bit[p];
    return idx;
}

// Swizzle term: which thread-id bits are XORed onto the float4-slot index.
constexpr uint32_t swz_of_tid(int c, uint32_t tid)
{
    return c >= 5 ? (tid & 7u) : ((tid >> (5 - c)) & ((1u << (c - 2)) - 1u));
}

// Physical word address of logical index `idx` in the layout owned by reader view v.
constexpr uint32_t view_phys(const View& v, uint32_t idx)
{
    uint32_t reg = 0, tid = 0;
    for (int p = 0; p < v.n; ++p) {
        const uint32_t b = (idx >> v.bit[p]) & 1u;
        if (p < v.c) reg |= b << p; else tid |= b << (p - v.c);
    }
#if WHVI_PADDED
    return tid * ((1u << v.c) + 4u) + reg;
#else
    const uint32_t slot = (reg >> 2) ^ swz_of_tid(v.c, tid);
    return (tid << v.c) + (slot << 2) + (reg & 3u);
#endif
}

// view_phys is GF(2)-linear in idx, so phys(a ^ b) = phys(a) ^ phys(b); the writer uses
//   phys = phys(tid part) ^ phys(reg part)
// with the register part a compile-time constant.

// Is logical bit b butterflied in round `round` of a transform over bits [0,k)?  A bit
// is processed in the first round (of views vs[0..]) where it is a register bit.
constexpr bool bit_is_new(const View* vs, int round, int b)
{
    for (int r = 0; r < round; ++r)
        if (view_has(vs[r], vs[r].c, b)) return false;
    return view_has(vs[round], vs[round].c, b);
}

// Number of rounds (1..3) of FIRST, MID, LAST needed to cover bits [0,k).
constexpr int rounds_needed(int n, int c, int k)
{
    const View vs[3] = {view_first(n, c), view_mid(n, c), view_last(n, c)};
    for (int r = 1; r <= 3; ++r) {
        bool ok = true;
        for (int b = 0; b < k; ++b) {
            bool cov = false;
            for (int q = 0; q < r; ++q) cov = cov || view_has(vs[q], c, b);
            ok = ok && cov;
        }
        if (ok) return r;
    }
    return 99;
}

}  // namespace whvi
