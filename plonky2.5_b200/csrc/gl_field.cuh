// Goldilocks field p = 2^64 - 2^32 + 1 on the sm_100a 32-bit integer datapath.
//
// Replaces plonky2 field/src/goldilocks_field.rs (add/sub/mul/reduce128) — semantics per SURVEY.md A.1; the
// constants are the ones visible at /root/reference/src/p3/mod.rs:55 (modulus) and
// /root/reference/src/p3/extension.rs:149,155 (generator 7, 2^32-th root 1753635133440165772).
//
// Representation rules used by the kernels:
//   * "canonical"  : value in [0, p)
//   * "any"        : value in [0, 2^64) congruent to the element (what reduce128 yields)
//   mul()/sqr() accept "any" operands and return "any"; add()/sub() need canonical operands and return
//   canonical; add_any_c()/sub_any_c() take (any, canonical) and return "any".
#pragma once
#include <stdint.h>

namespace gl {

constexpr uint64_t P = 0xFFFFFFFF00000001ULL;
constexpr uint64_t EPS = 0xFFFFFFFFULL;  // 2^64 mod p

__host__ __device__ __forceinline__ uint64_t canon(uint64_t x) { return x >= P ? x - P : x; }

// (z3:z2:z1:z0) -> 64 bits ("any"):  2^64 = 2^32 - 1 and 2^96 = -1 (mod p), so the value is X - z3 + z2*(2^32 - 1) with
// X = (z1:z0).  The three 64-bit wrap-arounds (one borrow each from "- z3" and "- z2", one carry from "+ z2*2^32") are
// collected in d in {-1, 0, 1} and folded back once as d*(2^32 - 1); a second wrap is impossible (tools/word_model.py
// checks this instruction sequence against big-integer arithmetic).  Written in PTX because the data flow through the
// carry flag is what keeps this at 12 integer instructions; nvcc's C++ lowering needs ~17 (64-bit compares + selects).
__device__ __forceinline__ uint64_t reduce_words(uint32_t z0, uint32_t z1, uint32_t z2, uint32_t z3) {
    uint32_t l, h;
    asm("{\n\t.reg .u32 d, ds;\n\t"
        "sub.cc.u32  %0, %2, %5;\n\t"
        "subc.cc.u32 %1, %3, 0;\n\t"
        "subc.u32    d, 0, 0;\n\t"
        "sub.cc.u32  %0, %0, %4;\n\t"
        "subc.cc.u32 %1, %1, 0;\n\t"
        "subc.u32    d, d, 0;\n\t"
        "add.cc.u32  %1, %1, %4;\n\t"
        "addc.u32    d, d, 0;\n\t"
        "shr.s32     ds, d, 31;\n\t"
        "sub.cc.u32  %0, %0, d;\n\t"
        "subc.u32    %1, %1, ds;\n\t"
        "add.u32     %1, %1, d;\n\t"
        "}" : "=&r"(l), "=&r"(h) : "r"(z0), "r"(z1), "r"(z2), "r"(z3));
    return ((uint64_t)h << 32) | l;
}
// (A variant that forms "+ z2*(2^32-1)" with one IMAD.WIDE — 3 fewer alu instructions, 1 more on the fma pipe — measured slower.)
__device__ __forceinline__ uint64_t reduce128(uint64_t lo, uint64_t hi) {
    return reduce_words((uint32_t)lo, (uint32_t)(lo >> 32), (uint32_t)hi, (uint32_t)(hi >> 32));
}

// 64 x 64 -> 128 as four IMAD.WIDE.U32 (the only multiplier shape the sm_100 fma-heavy pipe has for integers: 32
// lanes/clk/SM) and five carry adds: (z3:z2:z1:z0) = a * b.
__device__ __forceinline__ void mul_words(uint64_t a, uint64_t b, uint32_t& z0, uint32_t& z1, uint32_t& z2, uint32_t& z3) {
    asm("{\n\t.reg .u64 p00, p01, p10, p11;\n\t.reg .u32 q0, q1, m0, m1, h0, h1;\n\t"
        "mul.wide.u32 p00, %4, %6;\n\t"
        "mul.wide.u32 p01, %4, %7;\n\t"
        "mul.wide.u32 p10, %5, %6;\n\t"
        "mul.wide.u32 p11, %5, %7;\n\t"
        "mov.b64 {%0, %1}, p00;\n\t"
        "mov.b64 {q0, q1}, p01;\n\t"
        "mov.b64 {m0, m1}, p10;\n\t"
        "mov.b64 {h0, h1}, p11;\n\t"
        "add.cc.u32  %1, %1, q0;\n\t"
        "addc.cc.u32 %2, h0, q1;\n\t"
        "addc.u32    %3, h1, 0;\n\t"
        "add.cc.u32  %1, %1, m0;\n\t"
        "addc.cc.u32 %2, %2, m1;\n\t"
        "addc.u32    %3, %3, 0;\n\t"
        "}" : "=&r"(z0), "=&r"(z1), "=&r"(z2), "=&r"(z3)
            : "r"((uint32_t)a), "r"((uint32_t)(a >> 32)), "r"((uint32_t)b), "r"((uint32_t)(b >> 32)));
}
// The same product through nvcc's 128-bit multiply (mul.lo.u64 + mul.hi.u64): ptxas then uses the carry-out / carry-in
// forms of IMAD.WIDE.U32 (which PTX cannot name), 4 IMAD.WIDE + IMAD.X + MOV + 1 IADD3 — one alu-pipe instruction
// instead of five.  Which form is faster depends on which pipe the surrounding code saturates (DESIGN.md §3).
__device__ __forceinline__ void mul_words_c(uint64_t a, uint64_t b, uint32_t& z0, uint32_t& z1, uint32_t& z2, uint32_t& z3) {
    const uint64_t lo = a * b, hi = __umul64hi(a, b);
    z0 = (uint32_t)lo; z1 = (uint32_t)(lo >> 32); z2 = (uint32_t)hi; z3 = (uint32_t)(hi >> 32);
}
#ifndef GL_MUL_NEW
#define GL_MUL_NEW 1
#endif
// "any" in, "any" out
__device__ __forceinline__ uint64_t mul(uint64_t a, uint64_t b) {
    uint32_t z0, z1, z2, z3;
#if GL_MUL_NEW
    mul_words_c(a, b, z0, z1, z2, z3);
#else
    mul_words(a, b, z0, z1, z2, z3);
#endif
    return reduce_words(z0, z1, z2, z3);
}
// a^2: the cross product a0*a1 is computed once and added twice (3 IMAD.WIDE.U32 instead of 4)
__device__ __forceinline__ uint64_t sqr(uint64_t a) {
    uint32_t z0, z1, z2, z3;
    asm("{\n\t.reg .u64 p00, p01, p11;\n\t.reg .u32 m0, m1, h0, h1;\n\t"
        "mul.wide.u32 p00, %4, %4;\n\t"
        "mul.wide.u32 p01, %4, %5;\n\t"
        "mul.wide.u32 p11, %5, %5;\n\t"
        "mov.b64 {%0, %1}, p00;\n\t"
        "mov.b64 {m0, m1}, p01;\n\t"
        "mov.b64 {h0, h1}, p11;\n\t"
        "add.cc.u32  %1, %1, m0;\n\t"
        "addc.cc.u32 %2, h0, m1;\n\t"
        "addc.u32    %3, h1, 0;\n\t"
        "add.cc.u32  %1, %1, m0;\n\t"
        "addc.cc.u32 %2, %2, m1;\n\t"
        "addc.u32    %3, %3, 0;\n\t"
        "}" : "=&r"(z0), "=&r"(z1), "=&r"(z2), "=&r"(z3) : "r"((uint32_t)a), "r"((uint32_t)(a >> 32)));
    return reduce_words(z0, z1, z2, z3);
}
__device__ __forceinline__ uint64_t mulc(uint64_t a, uint64_t b) { return canon(mul(a, b)); }

// canonical (+/-) canonical -> canonical
__device__ __forceinline__ uint64_t add(uint64_t a, uint64_t b) {
    uint64_t nb = P - b;                    // in (0, p]
    uint64_t d = a - nb;
    if (a < nb) d += P;
    return d;
}
__device__ __forceinline__ uint64_t sub(uint64_t a, uint64_t b) {
    uint64_t d = a - b;
    if (a < b) d += P;
    return d;
}
// any + canonical -> any
__device__ __forceinline__ uint64_t add_any_c(uint64_t a, uint64_t b) {
    uint64_t s = a + b;
    if (s < a) s += EPS;                    // a+b < 2^64 + p  =>  wrapped < p  =>  no second overflow
    return s;
}

// any + any -> any.  A 64-bit carry is worth 2^64 = 2^32 - 1; folding it can carry once more (only when the wrapped sum
// is >= p), never a third time.
__device__ __forceinline__ uint64_t add_any(uint64_t a, uint64_t b) {
    uint32_t l, h;
    asm("{\n\t.reg .u32 m;\n\t"
        "add.cc.u32  %0, %2, %4;\n\t"
        "addc.cc.u32 %1, %3, %5;\n\t"
        "addc.u32    m, 0, 0;\n\t"     // (subc after add.cc is NOT the carry: sm_100 keeps borrows as inverted carries)
        "neg.s32     m, m;\n\t"        // 0xFFFFFFFF * carry = (2^32 - 1) * carry
        "add.cc.u32  %0, %0, m;\n\t"
        "addc.cc.u32 %1, %1, 0;\n\t"
        "addc.u32    m, 0, 0;\n\t"
        "neg.s32     m, m;\n\t"
        "add.cc.u32  %0, %0, m;\n\t"
        "addc.u32    %1, %1, 0;\n\t"
        "}" : "=&r"(l), "=&r"(h) : "r"((uint32_t)a), "r"((uint32_t)(a >> 32)), "r"((uint32_t)b), "r"((uint32_t)(b >> 32)));
    return ((uint64_t)h << 32) | l;
}
// any - any -> any (a borrow is worth -(2^32 - 1); the fold can borrow once more, never a third time)
__device__ __forceinline__ uint64_t sub_any(uint64_t a, uint64_t b) {
    uint32_t l, h;
    asm("{\n\t.reg .u32 m;\n\t"
        "sub.cc.u32  %0, %2, %4;\n\t"
        "subc.cc.u32 %1, %3, %5;\n\t"
        "subc.u32    m, 0, 0;\n\t"
        "sub.cc.u32  %0, %0, m;\n\t"
        "subc.cc.u32 %1, %1, 0;\n\t"
        "subc.u32    m, 0, 0;\n\t"
        "sub.cc.u32  %0, %0, m;\n\t"
        "subc.u32    %1, %1, 0;\n\t"
        "}" : "=&r"(l), "=&r"(h) : "r"((uint32_t)a), "r"((uint32_t)(a >> 32)), "r"((uint32_t)b), "r"((uint32_t)(b >> 32)));
    return ((uint64_t)h << 32) | l;
}
// The quadratic extension F_p[X]/(X^2 - 7) (plonky2 field/src/extension/quadratic.rs; W = 7 as /root/reference/src/p3/extension.rs:147-151):
// an element is [a0, a1] = a0 + a1 X.  The one device F_p^2 product: FRI folding, openings and the extension gates use it.
struct Ext { uint64_t a0, a1; };
__device__ __forceinline__ Ext ext_mul(Ext a, Ext b) {   // canonical in/out
    uint64_t m00 = mulc(a.a0, b.a0), m11 = mulc(a.a1, b.a1);
    uint64_t m01 = mulc(a.a0, b.a1), m10 = mulc(a.a1, b.a0);
    Ext r;
    r.a0 = add(m00, mulc(m11, 7));
    r.a1 = add(m01, m10);
    return r;
}
__device__ __forceinline__ Ext ext_add(Ext a, Ext b) { return {add(a.a0, b.a0), add(a.a1, b.a1)}; }

// x * 2^24 and x * 2^48 (any -> any): the 8th and 4th roots of unity of plonky2's root choice are powers of two
// (w_8 = 2^120 = -2^24, w_4 = 2^48, w_8^3 = 2^168 = -2^72), so the radix-8 butterflies need shifts, not multiplies.
__device__ __forceinline__ uint64_t mul_2_24(uint64_t x) {
    const uint32_t x0 = (uint32_t)x, x1 = (uint32_t)(x >> 32);
    return reduce_words(x0 << 24, __funnelshift_l(x0, x1, 24), x1 >> 8, 0u);
}
__device__ __forceinline__ uint64_t mul_2_48(uint64_t x) {
    const uint32_t x0 = (uint32_t)x, x1 = (uint32_t)(x >> 32);
    return reduce_words(0u, x0 << 16, __funnelshift_l(x0, x1, 16), x1 >> 16);
}
// 2^72 = (2^32 - 1) * 2^8 (mod p)
__device__ __forceinline__ uint64_t mul_2_72(uint64_t x) { return mul(x, 0xFFFFFFFF00ULL); }

__host__ __device__ __forceinline__ uint32_t bitrev32(uint32_t x, uint32_t bits) {
#ifdef __CUDA_ARCH__
    return bits ? (__brev(x) >> (32 - bits)) : 0;
#else
    uint32_t r = 0;
    for (uint32_t i = 0; i < bits; i++) { r = (r << 1) | (x & 1); x >>= 1; }
    return r;
#endif
}

// ---- host-side helpers (table generation in the context; not on any hot path) -------------------------
__host__ inline uint64_t h_mul(uint64_t a, uint64_t b) {
    unsigned __int128 x = (unsigned __int128)a * b;
    uint64_t lo = (uint64_t)x, hi = (uint64_t)(x >> 64);
    uint64_t hh = hi >> 32, hl = hi & EPS;
    uint64_t t0 = lo - hh;
    if (lo < hh) t0 -= EPS;
    uint64_t t1 = hl * EPS;
    uint64_t t2 = t0 + t1;
    if (t2 < t0) t2 += EPS;
    return canon(t2);
}
__host__ inline uint64_t h_pow(uint64_t b, uint64_t e) {
    uint64_t r = 1;
    while (e) {
        if (e & 1) r = h_mul(r, b);
        b = h_mul(b, b);
        e >>= 1;
    }
    return r;
}
__host__ inline uint64_t h_inv(uint64_t a) { return h_pow(a, P - 2); }
constexpr uint64_t POWER_OF_TWO_GENERATOR = 1753635133440165772ULL;  // order 2^32
constexpr uint64_t COSET_SHIFT = 7;                                  // MULTIPLICATIVE_GROUP_GENERATOR
__host__ inline uint64_t h_root_of_unity(uint32_t n_log) { return h_pow(POWER_OF_TWO_GENERATOR, 1ULL << (32 - n_log)); }

}  // namespace gl
