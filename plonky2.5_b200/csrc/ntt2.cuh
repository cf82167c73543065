// K1/K2/K3, second generation: the batched Goldilocks NTT pass over the row-major matrix with
//   * 128-bit global and shared-memory accesses — a thread owns TWO adjacent columns of 8 tile rows in the radix-8 rounds (one
//     twiddle / pre-scale / index computation serves both columns), or one column of 16 tile rows in a radix-16 round;
//   * carry-save butterflies — a value in flight is three 32-bit words (l, h, t) = l + h*2^32 + t*2^64, unsigned with a small t, so an
//     add or a subtract is 3 carry-chain instructions instead of the 8-10 of a folded 64-bit modular add; a handful of inputs are
//     biased by a multiple of p up front so that no subtraction goes negative, the shift-multiplies take three-word inputs directly,
//     and values are folded back to 64 bits once per radix-8 / radix-16 step (8 instructions);
//   * an all-shift radix-16 last round — plonky2's roots of unity up to order 64 are powers of two (w_16 = 2^156 = -2^60, w_8 =
//     2^120 = -2^24, w_4 = 2^48), so the last four stages of a pass need no table twiddle at all.
// Same contract as ntt::ntt_pass_kernel (ntt.cuh): one pass = a 2^A-point DIF NTT on index bits [log_blk - A, log_blk), then the
// inter-pass twiddle if lower bits remain; same PassParams, same store modes.
//
// Replaces plonky2 field/src/fft.rs · fft_classic / ifft_with_options and field/src/polynomial/mod.rs · coset_fft_with_options
// (SURVEY.md A.2-A.4), driven from /root/reference/src/p3/mod.rs:250,260.  tools/ntt2_model.py mirrors every carry chain below on
// 32-bit words, checks it against big integers and PROVES the bias plan (no negative difference, third words within the funnel
// budgets) by interval propagation.
#pragma once
#include "ntt.cuh"

namespace ntt2 {

struct W3 { uint32_t l, h, t; };

__device__ __forceinline__ W3 w3(uint64_t x) { return {(uint32_t)x, (uint32_t)(x >> 32), 0u}; }

__device__ __forceinline__ W3 add3(const W3 a, const W3 b) {
    W3 r;
    asm("add.cc.u32  %0, %3, %6;\n\t"
        "addc.cc.u32 %1, %4, %7;\n\t"
        "addc.u32    %2, %5, %8;"
        : "=&r"(r.l), "=&r"(r.h), "=r"(r.t) : "r"(a.l), "r"(a.h), "r"(a.t), "r"(b.l), "r"(b.h), "r"(b.t));
    return r;
}
__device__ __forceinline__ W3 sub3(const W3 a, const W3 b) {   // a >= b (the bias plan guarantees it)
    W3 r;
    asm("sub.cc.u32  %0, %3, %6;\n\t"
        "subc.cc.u32 %1, %4, %7;\n\t"
        "subc.u32    %2, %5, %8;"
        : "=&r"(r.l), "=&r"(r.h), "=r"(r.t) : "r"(a.l), "r"(a.h), "r"(a.t), "r"(b.l), "r"(b.h), "r"(b.t));
    return r;
}
// a + K*p,  K*p = K + (2^32 - K)*2^32 + (K - 1)*2^64
template <uint32_t K>
__device__ __forceinline__ W3 bias3(const W3 a) {
    W3 r;
    asm("add.cc.u32  %0, %3, %6;\n\t"
        "addc.cc.u32 %1, %4, %7;\n\t"
        "addc.u32    %2, %5, %8;"
        : "=&r"(r.l), "=&r"(r.h), "=r"(r.t) : "r"(a.l), "r"(a.h), "r"(a.t), "n"(K), "n"(0u - K), "n"(K - 1));
    return r;
}
// (l, h, t) -> 64-bit "any": X + t*(2^32 - 1); one wrap at most, and after a wrap the value is tiny, so the second add cannot wrap
__device__ __forceinline__ uint64_t fold3(const W3 a) {
    uint32_t l, h;
    asm("{\n\t.reg .u32 u0, u1, c;\n\t"
        "sub.cc.u32  u0, 0, %4;\n\t"
        "subc.u32    u1, %4, 0;\n\t"
        "add.cc.u32  %0, %2, u0;\n\t"
        "addc.cc.u32 %1, %3, u1;\n\t"
        "addc.u32    c, 0, 0;\n\t"
        "neg.s32     c, c;\n\t"
        "add.cc.u32  %0, %0, c;\n\t"
        "addc.u32    %1, %1, 0;\n\t"
        "}" : "=&r"(l), "=&r"(h) : "r"(a.l), "r"(a.h), "r"(a.t));
    return ((uint64_t)h << 32) | l;
}
// (z2:z1:z0) -> 64-bit "any": X - z2 + z2*2^32 (reduce_words with z3 = 0)
__device__ __forceinline__ uint64_t reduce3(uint32_t z0, uint32_t z1, uint32_t z2) {
    uint32_t l, h;
    asm("{\n\t.reg .u32 d, ds;\n\t"
        "sub.cc.u32  %0, %2, %4;\n\t"
        "subc.cc.u32 %1, %3, 0;\n\t"
        "subc.u32    d, 0, 0;\n\t"
        "add.cc.u32  %1, %1, %4;\n\t"
        "addc.u32    d, d, 0;\n\t"
        "shr.s32     ds, d, 31;\n\t"
        "sub.cc.u32  %0, %0, d;\n\t"
        "subc.u32    %1, %1, ds;\n\t"
        "add.u32     %1, %1, d;\n\t"
        "}" : "=&r"(l), "=&r"(h) : "r"(z0), "r"(z1), "r"(z2));
    return ((uint64_t)h << 32) | l;
}
// a * 2^S mod p for a three-word a (t < 2^(32 - S%32)); S in {12, 24, 36, 48, 60, 72, 84}
template <int S>
__device__ __forceinline__ uint64_t shift_mul(const W3 a) {
    constexpr int R = S % 32, W = S / 32;
    static_assert(R > 0 && W <= 2, "unsupported shift");
    const uint32_t y0 = a.l << R, y1 = __funnelshift_l(a.l, a.h, R), y2 = __funnelshift_l(a.h, a.t, R);
    if (W == 0) return reduce3(y0, y1, y2);
    if (W == 1) return gl::reduce_words(0u, y0, y1, y2);
    // y * 2^64 = y * 2^32 - y: a non-negative four-word difference
    uint32_t r0, r1, r2, r3;
    asm("sub.cc.u32  %0, 0, %4;\n\t"
        "subc.cc.u32 %1, %4, %5;\n\t"
        "subc.cc.u32 %2, %5, %6;\n\t"
        "subc.u32    %3, %6, 0;"
        : "=&r"(r0), "=&r"(r1), "=&r"(r2), "=r"(r3) : "r"(y0), "r"(y1), "r"(y2));
    return gl::reduce_words(r0, r1, r2, r3);
}

// 8-point DIF on three-word inputs (natural order) -> 64-bit outputs in in-place-DIF order: out[e] = sum_j x_j w8^(j*bitrev3(e)).
// Bias plan K8 of tools/ntt2_model.py (x0: 22p, x2: 5p, x5: 10p, x7: 5p, a5: 2p), proved for inputs < 5 * 2^64.
__device__ __forceinline__ void dft8_cs(W3 (&x)[8], uint64_t (&out)[8]) {
    x[0] = bias3<22>(x[0]); x[2] = bias3<5>(x[2]); x[5] = bias3<10>(x[5]); x[7] = bias3<5>(x[7]);
    W3 a[8];
    a[0] = add3(x[0], x[4]); a[4] = sub3(x[0], x[4]);
    a[1] = add3(x[1], x[5]); a[5] = w3(shift_mul<24>(sub3(x[5], x[1])));   // (x1 - x5) * w8   = (x5 - x1) * 2^24
    a[2] = add3(x[2], x[6]); a[6] = w3(shift_mul<48>(sub3(x[2], x[6])));   // (x2 - x6) * w8^2
    a[3] = add3(x[3], x[7]); a[7] = w3(shift_mul<72>(sub3(x[7], x[3])));   // (x3 - x7) * w8^3 = (x7 - x3) * 2^72
    a[5] = bias3<2>(a[5]);
    W3 b[8];
    b[0] = add3(a[0], a[2]); b[2] = sub3(a[0], a[2]);
    b[1] = add3(a[1], a[3]); b[3] = w3(shift_mul<48>(sub3(a[1], a[3])));
    b[4] = add3(a[4], a[6]); b[6] = sub3(a[4], a[6]);
    b[5] = add3(a[5], a[7]); b[7] = w3(shift_mul<48>(sub3(a[5], a[7])));
    out[0] = fold3(add3(b[0], b[1])); out[1] = fold3(sub3(b[0], b[1]));
    out[2] = fold3(add3(b[2], b[3])); out[3] = fold3(sub3(b[2], b[3]));
    out[4] = fold3(add3(b[4], b[5])); out[5] = fold3(sub3(b[4], b[5]));
    out[6] = fold3(add3(b[6], b[7])); out[7] = fold3(sub3(b[6], b[7]));
}
__device__ __forceinline__ void dft8_cs(uint64_t (&x)[8]) {
    W3 v[8];
#pragma unroll
    for (int j = 0; j < 8; j++) v[j] = w3(x[j]);
    dft8_cs(v, x);
}

// 16-point DIF, all twiddles powers of two: w16^j = 2^(156 j mod 192): j=1: -2^60, 2: -2^24, 3: 2^84, 4: 2^48, 5: 2^12, 6: -2^72, 7: -2^36.
// In-place-DIF order: x[e] = sum_j x_j w16^(j*bitrev4(e)).
__device__ __forceinline__ void dft16_cs(uint64_t (&x)[16]) {
    W3 s[8], d[8];
    {
        const W3 x0 = bias3<2>(w3(x[0])), x8 = w3(x[8]);
        s[0] = add3(x0, x8); d[0] = sub3(x0, x8);
    }
#define NTT2_PAIR(J, SH, NEG)                                                                        \
    {                                                                                                \
        W3 lo = w3(x[J]), hi = w3(x[J + 8]);                                                         \
        if (NEG) { hi = bias3<2>(hi); s[J] = add3(lo, hi); d[J] = w3(shift_mul<SH>(sub3(hi, lo))); } \
        else { lo = bias3<2>(lo); s[J] = add3(lo, hi); d[J] = w3(shift_mul<SH>(sub3(lo, hi))); }     \
    }
    NTT2_PAIR(1, 60, true) NTT2_PAIR(2, 24, true) NTT2_PAIR(3, 84, false) NTT2_PAIR(4, 48, false)
    NTT2_PAIR(5, 12, false) NTT2_PAIR(6, 72, true) NTT2_PAIR(7, 36, true)
#undef NTT2_PAIR
    uint64_t lo8[8], hi8[8];
    dft8_cs(s, lo8);
    dft8_cs(d, hi8);
#pragma unroll
    for (int j = 0; j < 8; j++) { x[j] = lo8[j]; x[j + 8] = hi8[j]; }
}

// ---- TMA bulk copy (cp.async.bulk, the non-tensor form) + mbarrier: the round-twiddle table of a pass is one contiguous block in
// global memory, so a single elected thread hands the whole copy to the TMA unit and every thread later waits on the mbarrier's phase.
// (The TILE itself is not moved by TMA: its rows are 2^b_lo rows apart, the first round consumes the loads straight from registers,
// and the pass is bound by the integer ALU pipe — ncu: alu 75-80 %, math-pipe throttle 3.6-3.9 warps per issue vs long scoreboard
// 0.5-1.8, DRAM 21-26 % — so staging the tile through shared memory would add LDS instructions without hiding anything; DESIGN.md §3.2.)
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
    const uint32_t b = (uint32_t)__cvta_generic_to_shared(bar);
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(b), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(b) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    const uint32_t b = (uint32_t)__cvta_generic_to_shared(bar);
    asm volatile("{\n\t.reg .pred p;\n\t"
                 "WAIT_%=:\n\t"
                 "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
                 "@p bra DONE_%=;\n\t"
                 "bra WAIT_%=;\n\t"
                 "DONE_%=:\n\t}" ::"r"(b), "r"(parity) : "memory");
}

// ---- pass structure ------------------------------------------------------------------------------------------------------------------------
// rounds of a 2^A-point pass: non-final rounds are radix-8 (radix-16 for A = 8) followed by a table twiddle; the final round is the
// all-shift radix-16 where the stage count allows it
__host__ __device__ constexpr int plan_n(int A) { return A >= 9 ? 3 : (A >= 5 ? 2 : 1); }
__host__ __device__ constexpr int plan_k(int A, int r) {
    switch (A) {
        case 3: return r == 0 ? 3 : 0;
        case 4: return r == 0 ? 4 : 0;
        case 5: return r == 0 ? 3 : (r == 1 ? 2 : 0);
        case 6: return r < 2 ? 3 : 0;
        case 7: return r == 0 ? 3 : (r == 1 ? 4 : 0);
        case 8: return r < 2 ? 4 : 0;
        case 9: return r < 3 ? 3 : 0;
        case 10: return r < 2 ? 3 : (r == 2 ? 4 : 0);
        default: return 0;
    }
}

__device__ __forceinline__ uint32_t insk(uint32_t q, uint32_t sh, uint32_t e, uint32_t k) {
    return ((q >> sh) << (sh + k)) | (e << sh) | (q & ((1u << sh) - 1));
}
__host__ __device__ constexpr uint32_t brev_const(uint32_t e, int k) {
    uint32_t r = 0;
    for (int i = 0; i < k; i++) r |= ((e >> i) & 1u) << (k - 1 - i);
    return r;
}

template <int A>
__host__ __device__ constexpr int pad_shift() { return plan_k(A, plan_n(A) - 1) == 4 ? 4 : 3; }   // stride of the final round's rows
template <int A, int G>
__host__ __device__ constexpr size_t smem_words() { return (size_t)((1u << A) + ((1u << A) >> pad_shift<A>())) * G + (1u << A); }

// one finished element: inter-pass twiddle / scale / canonicalisation, then the store of its mode (see ntt::PassParams)
// inter-pass twiddle w_{2^log_blk}^(o_lo * bitrev_a(l)) of tile row l, looked up in W (w_N^e, e < N/2); only when lower bits remain
__device__ __forceinline__ uint64_t inter_twiddle(const ntt::PassParams& p, uint32_t l, uint32_t a, uint32_t o_lo) {
    const uint32_t N = 1u << p.log_n;
    const uint32_t ex = (o_lo * gl::bitrev32(l, a)) << (p.log_n - p.log_blk);
    return ex >= (N >> 1) ? gl::P - __ldg(p.W + (ex - (N >> 1))) : __ldg(p.W + ex);
}
__device__ __forceinline__ uint64_t finish(const ntt::PassParams& p, uint64_t v, uint64_t w, uint32_t b_lo) {
    if (b_lo) v = gl::mul(v, w);
    if (p.scale != 1) v = gl::mul(v, p.scale);
    if (!b_lo) v = gl::canon(v);   // only what leaves the NTT is canonical; between passes any 64-bit representative will do
    return v;
}
__device__ __forceinline__ uint64_t* dest(const ntt::PassParams& p, uint32_t prow, uint32_t col) {
    if (p.store_mode == 2) {
        const uint64_t grow = p.scatter_row0 + prow;
        return p.peer[grow >> p.log_rows_per_peer] + (grow & ((1ULL << p.log_rows_per_peer) - 1)) * p.scatter_pitch + p.scatter_col0 + col;
    }
    const uint32_t N = 1u << p.log_n;
    const uint32_t drow = p.store_mode == 1 ? ((N - gl::bitrev32(prow, p.log_n)) & (N - 1)) : prow;
    return p.dst + (uint64_t)drow * p.dst_pitch + col;
}

// G columns per tile (4 or 8), 2^A rows; (2^A * G) / 16 threads, 16 elements each
template <int G, int A>
__global__ void __launch_bounds__((1 << A) * G / 16 >= 32 ? (1 << A) * G / 16 : 32,
                                   (1 << A) * G / 16 >= 32 ? 1024 / ((1 << A) * G / 16) : 32)   // 1024 threads per SM => <= 64 registers
ntt_pass_kernel(const ntt::PassParams p) {
    constexpr int NR = plan_n(A);
    constexpr uint32_t T = 1u << A, G2 = G / 2, PAD = pad_shift<A>();
    extern __shared__ __align__(128) uint64_t sm2[];
    __shared__ uint64_t wl_bar;                               // mbarrier of the twiddle-table bulk copy
    uint64_t* tile = sm2;                                     // [T + T/2^PAD][G]
    uint64_t* Wl = sm2 + (size_t)(T + (T >> PAD)) * G;        // w_T^j, j < T
    const uint32_t tid = threadIdx.x;
    // launched with exactly T * G / 16 threads: every thread owns 16 elements of the tile
    const uint32_t cg = blockIdx.x % p.ncg, tile_id = blockIdx.x / p.ncg;
    const uint32_t b_lo = p.log_blk - A;
    const uint32_t o_lo = tile_id & ((1u << b_lo) - 1), o_hi = tile_id >> b_lo;
    const uint32_t row_base = (o_hi << p.log_blk) | o_lo;
    auto phys = [](uint32_t l) { return l + (l >> PAD); };
    // two mappings of the tile onto the threads: 8 rows x 2 columns (radix-8 rounds) or 16 rows x 1 column (radix-16 rounds)
    const uint32_t q8 = tid / G2, c2 = tid % G2, q16 = tid / G, c1 = tid % G;
    const uint32_t col2 = cg * G + 2 * c2, col1 = cg * G + c1;
    const uint64_t* const src = p.src_list ? p.peer[cg] - (size_t)cg * G : p.src;   // one block per column group, or one matrix

    if (NR > 1) {
        if (tid == 0) mbar_init(&wl_bar, 1);
        __syncthreads();                                      // the initialised barrier is visible to every waiter
    }
    ulonglong2 v[8];     // radix-8 view: v[e] = columns (col2, col2 + 1) of tile row insk(q8, sh, e, 3)
    uint64_t u[16];      // radix-16 view: u[e] = column col1 of tile row insk(q16, sh, e, 4)
    constexpr int K0 = plan_k(A, 0);
    constexpr uint32_t SH0 = A - K0;
    {
        if (K0 == 3) {
#pragma unroll
            for (int e = 0; e < 8; e++) {
                const uint64_t row = row_base | ((uint64_t)insk(q8, SH0, e, 3) << b_lo);
                v[e] = *reinterpret_cast<const ulonglong2*>(src + row * p.src_pitch + col2);
            }
        } else {
#pragma unroll
            for (int e = 0; e < 16; e++) {
                const uint64_t row = row_base | ((uint64_t)insk(q16, SH0, e, 4) << b_lo);
                u[e] = src[row * p.src_pitch + col1];
            }
        }
    }
    // (the tile's own loads were issued above; the table copy now runs on the TMA unit in their shadow)
    if (NR > 1 && tid == 0) tma_bulk_g2s(Wl, p.Wa, T * 8, &wl_bar);
    if (p.pre != nullptr) {
        if (K0 == 3) {
#pragma unroll
            for (int e = 0; e < 8; e++) {
                const uint64_t row = row_base | ((uint64_t)insk(q8, SH0, e, 3) << b_lo);
                const uint64_t g = __ldg(p.pre + row);
                v[e].x = gl::mul(v[e].x, g);
                v[e].y = gl::mul(v[e].y, g);
            }
        } else {
#pragma unroll
            for (int e = 0; e < 16; e++) {
                const uint64_t row = row_base | ((uint64_t)insk(q16, SH0, e, 4) << b_lo);
                u[e] = gl::mul(u[e], __ldg(p.pre + row));
            }
        }
    }
    if (NR > 1) mbar_wait(&wl_bar, 0);   // Wl has landed (phase 0 of the mbarrier completes when all T*8 bytes have arrived)

    int done = 0;
#pragma unroll
    for (int r = 0; r < NR; r++) {
        const int k = plan_k(A, r);
        const uint32_t sh = A - done - k;          // tile bit of this round's local bit 0
        const bool last = r + 1 == NR;
        if (r > 0) {
            // exchange: the previous round's elements go to the tile, this round's come back
            const int kp = plan_k(A, r - 1);
            const uint32_t shp = A - done;
            {
                if (kp == 3) {
#pragma unroll
                    for (int e = 0; e < 8; e++)
                        *reinterpret_cast<ulonglong2*>(tile + (size_t)phys(insk(q8, shp, e, 3)) * G + 2 * c2) = v[e];
                } else {
#pragma unroll
                    for (int e = 0; e < 16; e++) tile[(size_t)phys(insk(q16, shp, e, 4)) * G + c1] = u[e];
                }
            }
            __syncthreads();
            {
                if (k == 4) {
#pragma unroll
                    for (int e = 0; e < 16; e++) u[e] = tile[(size_t)phys(insk(q16, sh, e, 4)) * G + c1];
                } else {   // 3 stages, or the 2-stage tail of A = 5 (held in the radix-8 layout at shift 0)
#pragma unroll
                    for (int e = 0; e < 8; e++)
                        v[e] = *reinterpret_cast<const ulonglong2*>(tile + (size_t)phys(insk(q8, k == 3 ? sh : 0, e, 3)) * G + 2 * c2);
                }
            }
            if (!last) __syncthreads();            // the tile is rewritten by the next exchange
        }
        {
            if (k == 4) {
                dft16_cs(u);
                if (!last) {
                    const uint32_t step = (q16 & ((1u << sh) - 1)) << (A - sh - 4);
#pragma unroll
                    for (int e = 1; e < 16; e++) u[e] = gl::mul(u[e], Wl[step * brev_const(e, 4)]);
                }
            } else if (k == 3) {
                uint64_t x[8], y[8];
#pragma unroll
                for (int e = 0; e < 8; e++) { x[e] = v[e].x; y[e] = v[e].y; }
                dft8_cs(x);
                dft8_cs(y);
                if (!last) {
                    const uint32_t step = (q8 & ((1u << sh) - 1)) << (A - sh - 3);
#pragma unroll
                    for (int e = 1; e < 8; e++) {
                        const uint64_t w = Wl[step * brev_const(e, 3)];
                        x[e] = gl::mul(x[e], w);
                        y[e] = gl::mul(y[e], w);
                    }
                }
#pragma unroll
                for (int e = 0; e < 8; e++) v[e] = make_ulonglong2(x[e], y[e]);
            } else {   // k == 2, final (A = 5): two radix-4 DFTs per column on local bits 1..0
                uint64_t x[8], y[8];
#pragma unroll
                for (int e = 0; e < 8; e++) { x[e] = v[e].x; y[e] = v[e].y; }
                ntt::radix8_round(x, Wl, A, 0, 0, 2);
                ntt::radix8_round(y, Wl, A, 0, 0, 2);
#pragma unroll
                for (int e = 0; e < 8; e++) v[e] = make_ulonglong2(x[e], y[e]);
            }
        }
        done += k;
    }
    // ---- the finished tile leaves: inter-pass twiddle / 1/N / canonical form, then the store of this pass's mode
    constexpr int KL = plan_k(A, NR - 1);
    if (KL == 4) {
        // the two shapes every LDE coset runs (16 of the 18 launches of a commit) without per-element mode branches: plain row-major
        // stores, no 1/N; the 16 rows of a thread are 2^b_lo rows apart, so one pointer walks them
        if (p.store_mode == 0 && p.scale == 1) {
            uint64_t* d = p.dst + (uint64_t)(row_base | ((q16 << 4) << b_lo)) * p.dst_pitch + col1;
            const uint64_t stride = (uint64_t)p.dst_pitch << b_lo;
            if (b_lo == 0) {
#pragma unroll
                for (int e = 0; e < 16; e++) d[e * stride] = gl::canon(u[e]);
            } else {
                // inter-pass twiddle w_{2^log_blk}^(o_lo * bitrev_A(l)), l = 16 q16 + e: bitrev_A(l) = bitrev_4(e) * 2^(A-4) + bitrev_(A-4)(q16)
                const uint32_t N = 1u << p.log_n, sh = p.log_n - p.log_blk;
                constexpr uint32_t A4 = A >= 4 ? A - 4 : 0;   // (this branch only exists for A >= 4)
                const uint32_t ex0 = (o_lo * gl::bitrev32(q16, A4)) << sh, exs = (o_lo << A4) << sh;
#pragma unroll
                for (int e = 0; e < 16; e++) {
                    const uint32_t ex = ex0 + exs * brev_const(e, 4);
                    const uint64_t w = ex >= (N >> 1) ? gl::P - __ldg(p.W + (ex - (N >> 1))) : __ldg(p.W + ex);
                    d[e * stride] = gl::mul(u[e], w);
                }
            }
            return;
        }
#pragma unroll
        for (int e = 0; e < 16; e++) {
            const uint32_t l = insk(q16, 0, e, 4);
            const uint64_t val = finish(p, u[e], b_lo ? inter_twiddle(p, l, A, o_lo) : 1, b_lo);
            if (p.store_mode == 2 && col1 >= p.scatter_ncols) continue;
            *dest(p, row_base | (l << b_lo), col1) = val;
        }
    } else {
#pragma unroll
        for (int e = 0; e < 8; e++) {
            const uint32_t l = insk(q8, 0, e, 3);
            const uint64_t w = b_lo ? inter_twiddle(p, l, A, o_lo) : 1;
            ulonglong2 val;
            val.x = finish(p, v[e].x, w, b_lo);
            val.y = finish(p, v[e].y, w, b_lo);
            uint64_t* d = dest(p, row_base | (l << b_lo), col2);
            if (p.store_mode == 2) {
                if (col2 + 1 < p.scatter_ncols && ((p.scatter_col0 | p.scatter_pitch) & 1) == 0) *reinterpret_cast<ulonglong2*>(d) = val;
                else {
                    if (col2 < p.scatter_ncols) d[0] = val.x;
                    if (col2 + 1 < p.scatter_ncols) d[1] = val.y;
                }
            } else {
                *reinterpret_cast<ulonglong2*>(d) = val;
            }
        }
    }
}

}  // namespace ntt2
