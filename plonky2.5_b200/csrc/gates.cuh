// §8(f) ranks 3-4: gate-constraint evaluation over the resident LDE rows, and witness generation, for the reference's own gates.
//
//   Poseidon2Gate           /root/reference/src/common/poseidon2/poseidon2_gate.rs:233-310 (eval_unfiltered_base_one: 135 wires ->
//                           123 constraints, degree 7) and :447-523 (Poseidon2Generator::run_once); the permutation pieces are
//                           /root/reference/src/common/poseidon2/poseidon2.rs:127-245 (matmul_external / matmul_m4 / matmul_internal)
//   U32ArithmeticGate       /root/reference/src/common/u32/gates/arithmetic_u32.rs:103-166 (num_ops x (4 + 32) constraints, degree 4)
//
// This is what plonky2 plonk/vanishing_poly.rs · evaluate_gate_constraints_base_batch does per gate inside compute_quotient_polys:
// one thread per LDE row (a leaf row of the wires commit, already in HBM), every constraint value multiplied by alpha_k^(offset + i)
// and accumulated per challenge k (plonk_common.rs · reduce_with_powers), optionally times a per-row filter value.
// All arithmetic is canonical Goldilocks (gl::add / gl::sub / gl::mulc): results are bit-exact field values.
#pragma once
#include "gl_field.cuh"
#include "poseidon2_constants.cuh"
#include "poseidon_constants.cuh"

namespace gates {

constexpr int P2_WIDTH = 12, P2_RF_BEGIN = 4, P2_RF_END = 8, P2_RP = 22;
constexpr int P2_WIRE_SWAP = 24, P2_START_DELTA = 25, P2_START_RF_BEGIN = 29, P2_START_PARTIAL = 29 + 12 * 3, P2_START_RF_END = 29 + 36 + 22;
constexpr int P2_NUM_WIRES = P2_START_RF_END + 12 * 4;                 // 135
constexpr int P2_NUM_CONSTRAINTS = 12 * 7 + 22 + 12 + 1 + 4;           // 123
constexpr int U32_LIMBS = 32, U32_ROUTED = 6;
constexpr int MAX_CONSTRAINTS = 160, MAX_CHALLENGES = 4;

struct PiHash { uint64_t w[4]; };   // the public-inputs hash (canonical), passed by value in the kernel arguments

__device__ __forceinline__ uint64_t dbl(uint64_t x) { return gl::add(x, x); }

__device__ __forceinline__ uint64_t sbox7(uint64_t x) {
    const uint64_t x2 = gl::sqr(x), x4 = gl::sqr(x2), x3 = gl::mul(x, x2);
    return gl::mulc(x3, x4);
}

// poseidon2.rs:185-245
__device__ __forceinline__ void matmul_m4(uint64_t (&s)[P2_WIDTH]) {
#pragma unroll
    for (int i = 0; i < 3; i++) {
        const int a = 4 * i;
        const uint64_t t0 = gl::add(s[a], s[a + 1]), t1 = gl::add(s[a + 2], s[a + 3]);
        const uint64_t t2 = gl::add(t1, dbl(s[a + 1])), t3 = gl::add(t0, dbl(s[a + 3]));
        const uint64_t t4 = gl::add(t3, dbl(dbl(t1))), t5 = gl::add(t2, dbl(dbl(t0)));
        s[a] = gl::add(t3, t5); s[a + 1] = t5; s[a + 2] = gl::add(t2, t4); s[a + 3] = t4;
    }
}
// poseidon2.rs:127-146
__device__ __forceinline__ void matmul_external(uint64_t (&s)[P2_WIDTH]) {
    matmul_m4(s);
    uint64_t st[4];
#pragma unroll
    for (int l = 0; l < 4; l++) st[l] = gl::add(gl::add(s[l], s[4 + l]), s[8 + l]);
#pragma unroll
    for (int i = 0; i < P2_WIDTH; i++) s[i] = gl::add(s[i], st[i & 3]);
}
// poseidon2.rs:164-182: s_i <- (MAT_DIAG_M_1[i] - 1) * s_i + sum(s)
__device__ __forceinline__ void matmul_internal(uint64_t (&s)[P2_WIDTH]) {
    uint64_t sum = s[0];
#pragma unroll
    for (int i = 1; i < P2_WIDTH; i++) sum = gl::add(sum, s[i]);
#pragma unroll
    for (int i = 0; i < P2_WIDTH; i++) s[i] = gl::add(gl::mulc(s[i], poseidon2::DIAG_M_2[i]), sum);
}

// The constraint stream of one Poseidon2Gate row, in the reference's order; `w(i)` reads wire i (canonical), `emit(v)` takes constraint values.
template <class Wires, class Emit>
__device__ __forceinline__ void poseidon2_gate(Wires&& w, Emit&& emit) {
    const uint64_t swap = w(P2_WIRE_SWAP);
    emit(gl::mulc(swap, gl::sub(swap, 1)));
    uint64_t s[P2_WIDTH];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const uint64_t lhs = w(i), rhs = w(i + 4), d = w(P2_START_DELTA + i);
        emit(gl::sub(gl::mulc(swap, gl::sub(rhs, lhs)), d));
        s[i] = gl::add(lhs, d);
        s[i + 4] = gl::sub(rhs, d);
    }
#pragma unroll
    for (int i = 8; i < P2_WIDTH; i++) s[i] = w(i);
    matmul_external(s);
#pragma unroll 1
    for (int r = 0; r < P2_RF_BEGIN; r++) {
#pragma unroll
        for (int i = 0; i < P2_WIDTH; i++) {
            uint64_t v = gl::add(s[i], poseidon2::RC[r][i]);
            if (r != 0) {
                const uint64_t in = w(P2_START_RF_BEGIN + P2_WIDTH * (r - 1) + i);
                emit(gl::sub(v, in));
                v = in;
            }
            s[i] = sbox7(v);
        }
        matmul_external(s);
    }
#pragma unroll 1
    for (int r = 0; r < P2_RP; r++) {
        const uint64_t v = gl::add(s[0], poseidon2::RC_MID[r]);
        const uint64_t in = w(P2_START_PARTIAL + r);
        emit(gl::sub(v, in));
        s[0] = sbox7(in);
        matmul_internal(s);
    }
#pragma unroll 1
    for (int r = P2_RF_BEGIN; r < P2_RF_END; r++) {
#pragma unroll
        for (int i = 0; i < P2_WIDTH; i++) {
            const uint64_t v = gl::add(s[i], poseidon2::RC[r][i]);
            const uint64_t in = w(P2_START_RF_END + P2_WIDTH * (r - P2_RF_BEGIN) + i);
            emit(gl::sub(v, in));
            s[i] = sbox7(in);
        }
        matmul_external(s);
    }
#pragma unroll
    for (int i = 0; i < P2_WIDTH; i++) emit(gl::sub(s[i], w(P2_WIDTH + i)));
}

// U32ArithmeticGate, eval_unfiltered order: per op [hi_not_max_or_lo_zero, combined - computed, 32 limb range products (j = 31..0), low, high]
template <class Wires, class Emit>
__device__ __forceinline__ void u32_arithmetic_gate(Wires&& w, Emit&& emit, uint32_t num_ops) {
    for (uint32_t i = 0; i < num_ops; i++) {
        const uint64_t m0 = w(6 * i), m1 = w(6 * i + 1), addend = w(6 * i + 2), lo = w(6 * i + 3), hi = w(6 * i + 4), inv = w(6 * i + 5);
        const uint64_t computed = gl::add(gl::mulc(m0, m1), addend);
        const uint64_t diff = gl::sub(0xFFFFFFFFULL, hi);
        const uint64_t hi_not_max = gl::sub(gl::mulc(inv, diff), 1);
        emit(gl::mulc(hi_not_max, lo));
        emit(gl::sub(gl::add(gl::mulc(hi, 1ULL << 32), lo), computed));
        uint64_t clo = 0, chi = 0;
#pragma unroll 1
        for (int j = U32_LIMBS - 1; j >= 0; j--) {
            const uint64_t limb = w(U32_ROUTED * num_ops + U32_LIMBS * i + j);
            uint64_t prod = limb;                                   // (limb - 0)
            prod = gl::mulc(prod, gl::sub(limb, 1));
            prod = gl::mulc(prod, gl::sub(limb, 2));
            prod = gl::mulc(prod, gl::sub(limb, 3));
            emit(prod);
            if (j < U32_LIMBS / 2) clo = gl::add(dbl(dbl(clo)), limb);
            else chi = gl::add(dbl(dbl(chi)), limb);
        }
        emit(gl::sub(clo, lo));
        emit(gl::sub(chi, hi));
    }
}

// ---- the reference's other u32 / b32 gates (/root/reference/src/common/u32/gates/*.rs · eval_unfiltered, same constraint order) -------
__device__ __forceinline__ uint64_t range4(uint64_t v) {   // v (v-1) (v-2) (v-3)
    return gl::mulc(gl::mulc(gl::mulc(v, gl::sub(v, 1)), gl::sub(v, 2)), gl::sub(v, 3));
}
__device__ __forceinline__ uint64_t range2(uint64_t v) { return gl::mulc(v, gl::sub(v, 1)); }
__device__ __forceinline__ uint64_t times4(uint64_t v) { return dbl(dbl(v)); }

// add_many_u32.rs:103-143; param = num_addends | num_ops << 8; 16 result limbs + 2 carry limbs of 2 bits
template <class Wires, class Emit>
__device__ __forceinline__ void add_many_gate(Wires&& w, Emit&& emit, uint32_t param) {
    const uint32_t na = param & 0xFF, num_ops = param >> 8, stride = na + 3;
    for (uint32_t i = 0; i < num_ops; i++) {
        uint64_t sum = w(stride * i + na);                                    // carry
        for (uint32_t j = 0; j < na; j++) sum = gl::add(sum, w(stride * i + j));
        const uint64_t res = w(stride * i + na + 1), car = w(stride * i + na + 2);
        emit(gl::sub(gl::add(gl::mulc(car, 1ULL << 32), res), sum));
        uint64_t rl = 0, cl = 0;
#pragma unroll 1
        for (int j = 17; j >= 0; j--) {
            const uint64_t limb = w(stride * num_ops + 18 * i + j);
            emit(range4(limb));
            if (j < 16) rl = gl::add(times4(rl), limb);
            else cl = gl::add(times4(cl), limb);
        }
        emit(gl::sub(rl, res));
        emit(gl::sub(cl, car));
    }
}
// subtraction_u32.rs:100-134; param = num_ops
template <class Wires, class Emit>
__device__ __forceinline__ void subtraction_gate(Wires&& w, Emit&& emit, uint32_t num_ops) {
    for (uint32_t i = 0; i < num_ops; i++) {
        const uint64_t x = w(5 * i), y = w(5 * i + 1), b = w(5 * i + 2), res = w(5 * i + 3), bo = w(5 * i + 4);
        const uint64_t initial = gl::sub(gl::sub(x, y), b);
        emit(gl::sub(res, gl::add(initial, gl::mulc(bo, 1ULL << 32))));
        uint64_t comb = 0;
#pragma unroll 1
        for (int j = 15; j >= 0; j--) {
            const uint64_t limb = w(5 * num_ops + 16 * i + j);
            emit(range4(limb));
            comb = gl::add(times4(comb), limb);
        }
        emit(gl::sub(comb, res));
        emit(gl::mulc(bo, gl::sub(1, bo)));
    }
}
// range_check_u32.rs:70-92; param = num_input_limbs
template <class Wires, class Emit>
__device__ __forceinline__ void range_check_gate(Wires&& w, Emit&& emit, uint32_t n) {
    for (uint32_t i = 0; i < n; i++) {
        uint64_t sum = 0;
        for (int j = 15; j >= 0; j--) sum = gl::add(times4(sum), w(n + 16 * i + j));   // reduce_with_powers(aux, 4)
        emit(gl::sub(sum, w(i)));
#pragma unroll 1
        for (int j = 0; j < 16; j++) emit(range4(w(n + 16 * i + j)));
    }
}
// interleave_u32.rs:104-140; param = num_ops; 32 big-endian bits per op
template <class Wires, class Emit>
__device__ __forceinline__ void interleave_gate(Wires&& w, Emit&& emit, uint32_t num_ops) {
    for (uint32_t i = 0; i < num_ops; i++) {
        const uint32_t b0 = 2 * num_ops + 32 * i;
        uint64_t v2 = 0, v4 = 0;
        for (int k = 0; k < 32; k++) {                                        // bits[0] is the most significant
            const uint64_t bit = w(b0 + k);
            v2 = gl::add(dbl(v2), bit);
            v4 = gl::add(times4(v4), bit);
        }
        emit(gl::sub(v2, w(2 * i)));
        emit(gl::sub(v4, w(2 * i + 1)));
#pragma unroll 1
        for (int k = 0; k < 32; k++) emit(range2(w(b0 + k)));
    }
}
// uninterleave_to_u32.rs:91-134 (B32 = false) / uninterleave_to_b32.rs:115-168 (B32 = true); param = num_ops; 64 big-endian bits per op
template <bool B32, class Wires, class Emit>
__device__ __forceinline__ void uninterleave_gate(Wires&& w, Emit&& emit, uint32_t num_ops) {
    for (uint32_t i = 0; i < num_ops; i++) {
        const uint32_t b0 = 3 * num_ops + 64 * i;
        uint64_t v2 = 0, ce = 0, co = 0;
        for (int k = 0; k < 64; k++) v2 = gl::add(dbl(v2), w(b0 + k));
        for (int j = 0; j < 32; j++) {                                        // Horner over j: coefficient 2^(31-j) or 4^(31-j)
            ce = gl::add(B32 ? times4(ce) : dbl(ce), w(b0 + 2 * j));
            co = gl::add(B32 ? times4(co) : dbl(co), w(b0 + 2 * j + 1));
        }
        emit(gl::sub(v2, w(3 * i)));
        emit(gl::sub(ce, w(3 * i + 1)));
        emit(gl::sub(co, w(3 * i + 2)));
#pragma unroll 1
        for (int k = 0; k < 64; k++) emit(range2(w(b0 + k)));
    }
}
// comparison.rs:112-190; param = num_bits | num_chunks << 8
template <class Wires, class Emit>
__device__ __forceinline__ void comparison_gate(Wires&& w, Emit&& emit, uint32_t param) {
    const uint32_t num_bits = param & 0xFF, nc = param >> 8, chunk_bits = (num_bits + nc - 1) / nc;
    const uint64_t base = 1ULL << chunk_bits;
    uint64_t f = 0, s = 0;
    for (int i = (int)nc - 1; i >= 0; i--) {
        f = gl::add(gl::mulc(f, base), w(4 + i));
        s = gl::add(gl::mulc(s, base), w(4 + nc + i));
    }
    emit(gl::sub(f, w(0)));
    emit(gl::sub(s, w(1)));
    uint64_t msd = 0;
    for (uint32_t i = 0; i < nc; i++) {
        const uint64_t fc = w(4 + i), sc = w(4 + nc + i);
        uint64_t pf = 1, ps = 1;
        for (uint64_t x = 0; x < base; x++) { pf = gl::mulc(pf, gl::sub(fc, x)); ps = gl::mulc(ps, gl::sub(sc, x)); }
        emit(pf);
        emit(ps);
        const uint64_t diff = gl::sub(sc, fc), dummy = w(4 + 2 * nc + i), eq = w(4 + 3 * nc + i), inter = w(4 + 4 * nc + i);
        emit(gl::sub(gl::mulc(diff, dummy), gl::sub(1, eq)));
        emit(gl::mulc(eq, diff));
        emit(gl::sub(inter, gl::mulc(eq, msd)));
        msd = gl::add(inter, gl::mulc(gl::sub(1, eq), diff));
    }
    emit(gl::sub(w(3), msd));
    uint64_t comb = 0;
    for (uint32_t k = 0; k <= chunk_bits; k++) {
        const uint64_t bit = w(4 + 5 * nc + k);
        emit(gl::mulc(bit, gl::sub(1, bit)));
    }
    for (int k = (int)chunk_bits; k >= 0; k--) comb = gl::add(dbl(comb), w(4 + 5 * nc + k));
    emit(gl::sub(gl::add(base, w(3)), comb));
    emit(gl::sub(w(2), w(4 + 5 * nc + chunk_bits)));
}

// ---- plonky2's core gates (plonky2 @ 3de92d9 gates/{noop,constant,public_input,arithmetic_base,base_sum}.rs · eval_unfiltered, same
// constraint order).  Upstream source is not in this tree: restated, parity unpinned (oracle/plonky2_gates_oracle.py restates the same
// items independently).  `k(j)` reads gate constant j (local_constants after remove_prefix), `pi` is the 4-word public-inputs hash.
// NoopGate has no constraints and is never evaluated.

// ConstantGate: param = num_consts; k(i) - w(i)
template <class Wires, class Consts, class Emit>
__device__ __forceinline__ void constant_gate(Wires&& w, Consts&& k, Emit&& emit, uint32_t n) {
    for (uint32_t i = 0; i < n; i++) emit(gl::sub(k(i), w(i)));
}
// PublicInputGate: w(i) - public_inputs_hash[i]
template <class Wires, class Emit>
__device__ __forceinline__ void public_input_gate(Wires&& w, const uint64_t (&pi)[4], Emit&& emit) {
#pragma unroll
    for (int i = 0; i < 4; i++) emit(gl::sub(w(i), pi[i]));
}
// ArithmeticGate (base field): param = num_ops; output - (k(0) m0 m1 + k(1) addend), wires [m0, m1, addend, output] per op
template <class Wires, class Consts, class Emit>
__device__ __forceinline__ void arithmetic_gate(Wires&& w, Consts&& k, Emit&& emit, uint32_t num_ops) {
    const uint64_t c0 = k(0), c1 = k(1);
    for (uint32_t i = 0; i < num_ops; i++) {
        const uint64_t computed = gl::add(gl::mulc(gl::mulc(w(4 * i), w(4 * i + 1)), c0), gl::mulc(w(4 * i + 2), c1));
        emit(gl::sub(w(4 * i + 3), computed));
    }
}
// BaseSumGate<B>: param = num_limbs | B << 8; reduce_with_powers(limbs, B) - sum, then prod_{v < B} (limb - v) per limb
template <class Wires, class Emit>
__device__ __forceinline__ void base_sum_gate(Wires&& w, Emit&& emit, uint32_t param) {
    const uint32_t n = param & 0xFF, base = param >> 8;
    uint64_t sum = 0;
    for (int j = (int)n - 1; j >= 0; j--) sum = gl::add(gl::mulc(sum, base), w(1 + j));
    emit(gl::sub(sum, w(0)));
#pragma unroll 1
    for (uint32_t j = 0; j < n; j++) {
        const uint64_t limb = w(1 + j);
        uint64_t prod = limb;
        for (uint32_t v = 1; v < base; v++) prod = gl::mulc(prod, gl::sub(limb, v));
        emit(prod);
    }
}

// ---- three more base-field gates of plonky2 @ 3de92d9 (gates/{poseidon,exponentiation,random_access}.rs · eval_unfiltered, same
// constraint order).  Upstream source is not in this tree: restated, parity unpinned (tests/plonky2_std_gates_oracle.py restates them too).

// coefficient i of output row r of plonky2's Poseidon MDS matrix: CIRC[i] + DIAG[r] at i = 0
__device__ __forceinline__ constexpr uint32_t mds_coeff(uint32_t i, uint32_t r) {
    constexpr uint32_t CIRC[P2_WIDTH] = {17, 15, 41, 16, 2, 28, 13, 13, 39, 18, 34, 20};
    return CIRC[i] + (r == 0 && i == 0 ? 8 : 0);
}
// L + H 2^32 < 2^74 as (H >> 32 + carry : x), reduced once
__device__ __forceinline__ uint64_t reduce_halves(uint64_t L, uint64_t H) {
    const uint64_t x = L + (H << 32);
    return gl::canon(gl::reduce128(x, (H >> 32) + (x < L)));
}
// plonky2 Poseidon::mds_layer: out[r] = sum_i CIRC[i] s[(i + r) % 12] + DIAG[r] s[r] (hash/poseidon_goldilocks.rs MDS_MATRIX_CIRC /
// MDS_MATRIX_DIAG, DIAG = 8 at r = 0 only).  The coefficients are small (sum 264 < 2^9), so the 32-bit halves of the canonical inputs
// are accumulated apart (each sum < 2^41, one IMAD.WIDE.U32 per term) and every lane is reduced once.
__device__ __forceinline__ void poseidon_mds(uint64_t (&s)[P2_WIDTH]) {
    uint32_t lo[P2_WIDTH], hi[P2_WIDTH];
#pragma unroll
    for (int i = 0; i < P2_WIDTH; i++) { lo[i] = (uint32_t)s[i]; hi[i] = (uint32_t)(s[i] >> 32); }
#pragma unroll
    for (int r = 0; r < P2_WIDTH; r++) {
        uint64_t L = 0, H = 0;
#pragma unroll
        for (int i = 0; i < P2_WIDTH; i++) {
            const uint32_t c = mds_coeff(i, r);
            L += (uint64_t)lo[(i + r) % P2_WIDTH] * c;
            H += (uint64_t)hi[(i + r) % P2_WIDTH] * c;
        }
        s[r] = reduce_halves(L, H);
    }
}

// plonky2 Poseidon::poseidon in the naive form (full_rounds / partial_rounds_naive, ALL_ROUND_CONSTANTS) from the state after the swap.
// `at(wire, v)` gets every S-box input PoseidonGate stores (the wire that holds it, the value computed from the state) and returns the
// value the S-box takes: the constraint stream emits v - wire and continues from the wire, the witness generator writes v.  The
// upstream gate writes the partial rounds in the "fast" form; it yields the same lane-0 S-box inputs, so the same constraints
// (DESIGN.md §3.4).
template <class At>
__device__ __forceinline__ void poseidon_rounds(uint64_t (&s)[P2_WIDTH], At&& at) {
#pragma unroll 1
    for (int r = 0; r < 4; r++) {
#pragma unroll
        for (int i = 0; i < P2_WIDTH; i++) {
            uint64_t v = gl::add(s[i], POSEIDON_RC[P2_WIDTH * r + i]);
            if (r != 0) v = at(P2_START_RF_BEGIN + P2_WIDTH * (r - 1) + i, v);
            s[i] = sbox7(v);
        }
        poseidon_mds(s);
    }
#pragma unroll 1
    for (int r = 0; r < P2_RP; r++) {
#pragma unroll
        for (int i = 0; i < P2_WIDTH; i++) s[i] = gl::add(s[i], POSEIDON_RC[P2_WIDTH * (4 + r) + i]);
        s[0] = sbox7(at(P2_START_PARTIAL + r, s[0]));
        poseidon_mds(s);
    }
#pragma unroll 1
    for (int r = 0; r < 4; r++) {
#pragma unroll
        for (int i = 0; i < P2_WIDTH; i++)
            s[i] = sbox7(at(P2_START_RF_END + P2_WIDTH * r + i, gl::add(s[i], POSEIDON_RC[P2_WIDTH * (26 + r) + i])));
        poseidon_mds(s);
    }
}

// PoseidonGate (gates/poseidon.rs): Poseidon2Gate's wire layout and constraint order — swap binary, 4 deltas, the S-box inputs of full
// rounds 1..3, of the 22 partial rounds and of the 4 second-half full rounds, then the 12 outputs (123 constraints, degree 7)
template <class Wires, class Emit>
__device__ __forceinline__ void poseidon_gate(Wires&& w, Emit&& emit) {
    const uint64_t swap = w(P2_WIRE_SWAP);
    emit(gl::mulc(swap, gl::sub(swap, 1)));
    uint64_t s[P2_WIDTH];
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const uint64_t lhs = w(i), rhs = w(i + 4), d = w(P2_START_DELTA + i);
        emit(gl::sub(gl::mulc(swap, gl::sub(rhs, lhs)), d));
        s[i] = gl::add(lhs, d);
        s[i + 4] = gl::sub(rhs, d);
    }
#pragma unroll
    for (int i = 8; i < P2_WIDTH; i++) s[i] = w(i);
    poseidon_rounds(s, [&](int wire, uint64_t v) {
        const uint64_t in = w(wire);
        emit(gl::sub(v, in));
        return in;
    });
#pragma unroll
    for (int i = 0; i < P2_WIDTH; i++) emit(gl::sub(s[i], w(P2_WIDTH + i)));
}

// ExponentiationGate (gates/exponentiation.rs): param = num_power_bits n; wires base 0, bits 1..n (little-endian), output 1+n,
// intermediates 2+n..1+2n.  For i < n, with prev = 1 (i = 0) or intermediate[i-1]^2 and b = bits[n-1-i]:
// prev (b base + 1 - b) - intermediate[i]; then output - intermediate[n-1]
template <class Wires, class Emit>
__device__ __forceinline__ void exponentiation_gate(Wires&& w, Emit&& emit, uint32_t n) {
    const uint64_t base = w(0);
    uint64_t prev = 1;
#pragma unroll 1
    for (uint32_t i = 0; i < n; i++) {
        const uint64_t b = w(n - i), inter = w(2 + n + i);
        emit(gl::sub(gl::mulc(prev, gl::add(gl::mulc(b, base), gl::sub(1, b))), inter));
        prev = gl::canon(gl::sqr(inter));
    }
    emit(gl::sub(w(1 + n), w(1 + 2 * n)));
}

// RandomAccessGate (gates/random_access.rs): param = bits | num_copies << 8 | num_extra_constants << 16, v = 2^bits.  Copy c: index at
// (2+v)c, claimed element (2+v)c+1, list (2+v)c+2+i; extra constant i at (2+v) num_copies + i; bit i of copy c at num_routed + c bits + i.
// Per copy: b(b-1) per bit, sum b_i 2^i - index, folded - claimed; then k(i) - extra_i.  The pairwise fold x + b(y - x) over the bits in
// order is the multilinear sum_i x_i prod_j (bit j of i ? b_j : 1 - b_j), evaluated term by term (exact field identity, no list buffer).
template <class Wires, class Consts, class Emit>
__device__ __forceinline__ void random_access_gate(Wires&& w, Consts&& k, Emit&& emit, uint32_t param) {
    const uint32_t bits = param & 0xFF, copies = (param >> 8) & 0xFF, extras = param >> 16, v = 1u << bits;
    const uint32_t extra0 = (2 + v) * copies, routed = extra0 + extras;
    for (uint32_t c = 0; c < copies; c++) {
        const uint32_t b0 = routed + c * bits, l0 = (2 + v) * c;
        uint64_t idx = 0;
        for (uint32_t j = 0; j < bits; j++) emit(range2(w(b0 + j)));
        for (int j = (int)bits - 1; j >= 0; j--) idx = gl::add(dbl(idx), w(b0 + j));
        emit(gl::sub(idx, w(l0)));
        uint64_t folded = 0;
#pragma unroll 1
        for (uint32_t i = 0; i < v; i++) {
            uint64_t t = w(l0 + 2 + i);
            for (uint32_t j = 0; j < bits; j++) {
                const uint64_t b = w(b0 + j);
                t = gl::mulc(t, (i >> j) & 1 ? b : gl::sub(1, b));
            }
            folded = gl::add(folded, t);
        }
        emit(gl::sub(folded, w(l0 + 1)));
    }
    for (uint32_t i = 0; i < extras; i++) emit(gl::sub(k(i), w(extra0 + i)));
}

// ---- plonky2's extension-field gates (plonky2 @ 3de92d9 gates/{arithmetic_extension,multiplication_extension,reducing_extension}.rs ·
// eval_unfiltered, D = 2; restated, parity unpinned, tests/plonky2_ext_gates_oracle.py restates them too).  An extension value is the two
// wires [a0, a1]; every extension constraint is emitted as to_basefield_array(), component 0 first, so it is two base constraints.
template <class Wires>
__device__ __forceinline__ gl::Ext ext_wire(uint32_t i, Wires&& w) { return {w(i), w(i + 1)}; }
template <class Emit>
__device__ __forceinline__ void emit_ext_sub(gl::Ext a, gl::Ext b, Emit&& emit) {
    emit(gl::sub(a.a0, b.a0));
    emit(gl::sub(a.a1, b.a1));
}

// ArithmeticExtensionGate: param = num_ops; op i at wires 8i + [m0, m1, addend, output]: output - ((m0 m1) k(0) + addend k(1))
template <class Wires, class Consts, class Emit>
__device__ __forceinline__ void arithmetic_extension_gate(Wires&& w, Consts&& k, Emit&& emit, uint32_t num_ops) {
    const uint64_t c0 = k(0), c1 = k(1);
#pragma unroll 1
    for (uint32_t i = 0; i < num_ops; i++) {
        const gl::Ext p = gl::ext_mul(ext_wire(8 * i, w), ext_wire(8 * i + 2, w)), a = ext_wire(8 * i + 4, w);
        const gl::Ext computed = {gl::add(gl::mulc(p.a0, c0), gl::mulc(a.a0, c1)), gl::add(gl::mulc(p.a1, c0), gl::mulc(a.a1, c1))};
        emit_ext_sub(ext_wire(8 * i + 6, w), computed, emit);
    }
}
// MulExtensionGate: param = num_ops; op i at wires 6i + [m0, m1, output]: output - (m0 m1) k(0)
template <class Wires, class Consts, class Emit>
__device__ __forceinline__ void mul_extension_gate(Wires&& w, Consts&& k, Emit&& emit, uint32_t num_ops) {
    const uint64_t c0 = k(0);
#pragma unroll 1
    for (uint32_t i = 0; i < num_ops; i++) {
        const gl::Ext p = gl::ext_mul(ext_wire(6 * i, w), ext_wire(6 * i + 2, w));
        emit_ext_sub(ext_wire(6 * i + 4, w), {gl::mulc(p.a0, c0), gl::mulc(p.a1, c0)}, emit);
    }
}
// ReducingExtensionGate (D = 2) and ReducingGate (D = 1, base-field coefficients): param = num_coeffs n; output 0, alpha 2, old_acc 4,
// coefficient i at 6 + D i, accumulator i at 6 + D n + 2i for i < n - 1 and accumulator n - 1 is the output.  From acc = old_acc:
// acc alpha + coeff_i - acc_i, then acc = acc_i (the wire)
template <int D, class Wires, class Emit>
__device__ __forceinline__ void reducing_gate(Wires&& w, Emit&& emit, uint32_t n) {
    const gl::Ext alpha = ext_wire(2, w);
    gl::Ext acc = ext_wire(4, w);
#pragma unroll 1
    for (uint32_t i = 0; i < n; i++) {
        const gl::Ext acc_i = ext_wire(i + 1 < n ? 6 + D * n + 2 * i : 0, w);
        gl::Ext next = gl::ext_mul(acc, alpha);
        if constexpr (D == 2) next = gl::ext_add(next, ext_wire(6 + 2 * i, w));
        else next.a0 = gl::add(next.a0, w(6 + i));
        emit_ext_sub(next, acc_i, emit);
        acc = acc_i;
    }
}

// ---- the gates plonky2's recursive verifier adds (plonky2 @ 3de92d9 gates/{poseidon_mds,coset_interpolation}.rs · eval_unfiltered, D = 2;
// restated, parity unpinned, tests/plonky2_recursion_gates_oracle.py restates them too; ReducingGate is reducing_gate<1> above).

// PoseidonMdsGate: ext input i at wires 2i, ext output i at 24 + 2i (i < 12).  Per output row i, component by component:
// out_i - (sum_j CIRC[j] in_{(i+j) % 12} + DIAG[i] in_i), the constants as base scalars (poseidon_mds's matrix and its 32-bit-halves
// accumulation).  One row at a time from the wire reader, so no 12-wide state is held (24 constraints, degree 1)
template <class Wires, class Emit>
__device__ __forceinline__ void poseidon_mds_gate(Wires&& w, Emit&& emit) {
#pragma unroll 1
    for (uint32_t i = 0; i < P2_WIDTH; i++) {
        uint64_t L0 = 0, H0 = 0, L1 = 0, H1 = 0;
#pragma unroll
        for (uint32_t j = 0; j < P2_WIDTH; j++) {
            const uint32_t c = mds_coeff(j, i), at = 2 * ((i + j) % P2_WIDTH);
            const uint64_t x0 = w(at), x1 = w(at + 1);
            L0 += (uint64_t)(uint32_t)x0 * c; H0 += (x0 >> 32) * c;
            L1 += (uint64_t)(uint32_t)x1 * c; H1 += (x1 >> 32) * c;
        }
        emit(gl::sub(w(24 + 2 * i), reduce_halves(L0, H0)));
        emit(gl::sub(w(25 + 2 * i), reduce_halves(L1, H1)));
    }
}

// the 2^bits-th root of unity of plonky2's choice (primitive_root_of_unity), bits 0..5
__constant__ uint64_t COSET_INTERPOLATION_ROOTS[6] = {1ULL, 0xFFFFFFFF00000000ULL, 0x1000000000000ULL, 0xFFFFFFFEFF000001ULL,
                                                      0xEFFFFFFF00000001ULL, 0x3FFFFFFFC000ULL};

// CosetInterpolationGate: param = subgroup_bits | degree << 8, n = 2^subgroup_bits, k = (n - 2) / (degree - 1) intermediates.  Wires:
// shift 0 (base), value i at 1 + 2i (i < n), evaluation point 1 + 2n, evaluation value 3 + 2n; with s = 5 + 2n, intermediate eval i at
// s + 2i, intermediate prod i at s + 2(k + i), shifted evaluation point s + 4k.  Constraints: evaluation_point - shifted_point shift; then
// partial_interpolate over domain[0, degree) from (eval, prod) = (0, 1), and for each i < k: int_eval_i - eval, int_prod_i - prod, continuing
// from those two wires over domain[1 + (degree - 1)(i + 1), min(that + degree - 1, n)); last evaluation_value - eval.  One step, with
// t = z' - x_j: eval <- eval t + (v_j w_j) prod, prod <- prod t.  The domain is the subgroup, so the barycentric weight of x_j = omega^j is
// w_j = x_j / n exactly; the chunks are consecutive, so x_j is stepped by omega and no table is read
template <class Wires, class Emit>
__device__ __forceinline__ void coset_interpolation_gate(Wires&& w, Emit&& emit, uint32_t param) {
    const uint32_t bits = param & 0xFF, degree = param >> 8, n = 1u << bits, k = (n - 2) / (degree - 1), s = 5 + 2 * n;
    const uint64_t shift = w(0), omega = COSET_INTERPOLATION_ROOTS[bits], n_inv = gl::P - ((gl::P - 1) >> bits);
    const gl::Ext z = ext_wire(s + 4 * k, w);
    const gl::Ext point = ext_wire(1 + 2 * n, w);
    emit(gl::sub(point.a0, gl::mulc(z.a0, shift)));
    emit(gl::sub(point.a1, gl::mulc(z.a1, shift)));
    gl::Ext eval = {0, 0}, prod = {1, 0};
    uint64_t x = 1;
    uint32_t next = degree, inter = 0;   // the domain index that ends the current chunk, the intermediate pair it is checked against
#pragma unroll 1
    for (uint32_t j = 0; j < n; j++) {
        if (j == next) {
            const gl::Ext ie = ext_wire(s + 2 * inter, w), ip = ext_wire(s + 2 * (k + inter), w);
            emit_ext_sub(ie, eval, emit);
            emit_ext_sub(ip, prod, emit);
            eval = ie; prod = ip;
            next += degree - 1; inter++;
        }
        const gl::Ext t = {gl::sub(z.a0, x), z.a1};
        const uint64_t wj = gl::mulc(x, n_inv);
        const gl::Ext vw = {gl::mulc(w(1 + 2 * j), wj), gl::mulc(w(2 + 2 * j), wj)};
        eval = gl::ext_add(gl::ext_mul(eval, t), gl::ext_mul(vw, prod));
        prod = gl::ext_mul(prod, t);
        x = gl::mulc(x, omega);
    }
    emit_ext_sub(ext_wire(3 + 2 * n, w), eval, emit);
}

enum { GATE_POSEIDON2 = 0, GATE_U32_ARITHMETIC = 1, GATE_U32_ADD_MANY = 2, GATE_U32_SUBTRACTION = 3, GATE_U32_RANGE_CHECK = 4,
       GATE_U32_INTERLEAVE = 5, GATE_UNINTERLEAVE_TO_U32 = 6, GATE_UNINTERLEAVE_TO_B32 = 7, GATE_COMPARISON = 8, GATE_NOOP = 9,
       GATE_CONSTANT = 10, GATE_PUBLIC_INPUT = 11, GATE_ARITHMETIC = 12, GATE_BASE_SUM = 13, GATE_POSEIDON = 15, GATE_EXPONENTIATION = 16,
       GATE_RANDOM_ACCESS = 17, GATE_ARITHMETIC_EXTENSION = 19, GATE_MUL_EXTENSION = 20, GATE_REDUCING_EXTENSION = 21,
       GATE_COSET_INTERPOLATION = 23, GATE_REDUCING = 24, GATE_POSEIDON_MDS = 25 };

// every kind but GATE_POSEIDON, which has kernel instances of its own (inlined here it would raise the register count of every gate)
template <class Wires, class Consts, class Emit>
__device__ __forceinline__ void eval_gate(int kind, uint32_t param, Wires&& w, Consts&& k, const uint64_t (&pi)[4], Emit&& emit) {
    switch (kind) {
        case GATE_POSEIDON2: poseidon2_gate(w, emit); break;
        case GATE_U32_ARITHMETIC: u32_arithmetic_gate(w, emit, param); break;
        case GATE_U32_ADD_MANY: add_many_gate(w, emit, param); break;
        case GATE_U32_SUBTRACTION: subtraction_gate(w, emit, param); break;
        case GATE_U32_RANGE_CHECK: range_check_gate(w, emit, param); break;
        case GATE_U32_INTERLEAVE: interleave_gate(w, emit, param); break;
        case GATE_UNINTERLEAVE_TO_U32: uninterleave_gate<false>(w, emit, param); break;
        case GATE_UNINTERLEAVE_TO_B32: uninterleave_gate<true>(w, emit, param); break;
        case GATE_CONSTANT: constant_gate(w, k, emit, param); break;
        case GATE_PUBLIC_INPUT: public_input_gate(w, pi, emit); break;
        case GATE_ARITHMETIC: arithmetic_gate(w, k, emit, param); break;
        case GATE_BASE_SUM: base_sum_gate(w, emit, param); break;
        case GATE_EXPONENTIATION: exponentiation_gate(w, emit, param); break;
        case GATE_RANDOM_ACCESS: random_access_gate(w, k, emit, param); break;
        case GATE_ARITHMETIC_EXTENSION: arithmetic_extension_gate(w, k, emit, param); break;
        case GATE_MUL_EXTENSION: mul_extension_gate(w, k, emit, param); break;
        case GATE_REDUCING_EXTENSION: reducing_gate<2>(w, emit, param); break;
        case GATE_COSET_INTERPOLATION: coset_interpolation_gate(w, emit, param); break;
        case GATE_REDUCING: reducing_gate<1>(w, emit, param); break;
        case GATE_POSEIDON_MDS: poseidon_mds_gate(w, emit); break;
        case GATE_NOOP: break;
        default: comparison_gate(w, emit, param); break;
    }
}

// plonky2 gates/selectors.rs · UNUSED_SELECTOR (u32::MAX)
constexpr uint64_t UNUSED_SELECTOR = 0xFFFFFFFFULL;

// plonky2 gates/gate.rs · compute_filter(i, group, s, many_selectors): prod_{j in [start, end), j != i} (j - s) * (UNUSED_SELECTOR - s if many)
__device__ __forceinline__ uint64_t selector_filter(uint64_t s, uint32_t i, uint32_t start, uint32_t end, uint32_t many) {
    uint64_t f = many ? gl::sub(UNUSED_SELECTOR, s) : 1;
#pragma unroll 1
    for (uint32_t j = start; j < end; j++)
        if (j != i) f = gl::mulc(f, gl::sub(j, s));
    return f;
}

// every constraint of every row, uncombined (tests): out[row][i]; consts [n_rows][n_consts] (nullptr when the gate reads none)
__global__ void gate_constraints_kernel(int kind, uint32_t param, const uint64_t* __restrict__ rows, uint32_t pitch, uint64_t n_rows,
                                        uint32_t n_constraints, const uint64_t* __restrict__ consts, uint32_t n_consts, const PiHash pi,
                                        uint64_t* __restrict__ out) {
    const uint64_t row = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= n_rows) return;
    const uint64_t* r = rows + row * pitch;
    const uint64_t* c = consts + row * n_consts;
    uint64_t* o = out + row * n_constraints;
    uint32_t k = 0;
    auto wires = [&](int i) { return gl::canon(__ldg(r + i)); };
    auto emit = [&](uint64_t v) { o[k++] = v; };
    if (kind == GATE_POSEIDON) poseidon_gate(wires, emit);
    else eval_gate(kind, param, wires, [&](int i) { return gl::canon(__ldg(c + i)); }, pi.w, emit);
}

enum { FILTER_NONE = 0, FILTER_COLUMN = 1, FILTER_SELECTOR = 2 };

struct QuotientArgs {
    const uint64_t* rows;          // wires: [n_rows][pitch] (the leaf matrix of the wires commit)
    const uint64_t* filter;        // [n_rows][filter_pitch] matrix the filter is read from (FILTER_COLUMN / FILTER_SELECTOR), else nullptr
    uint64_t* acc;                 // [n_challenges][n_rows], += in place
    const uint64_t* powers;        // [n_challenges][n_constraints]: alpha_k^(offset + i), canonical
    uint64_t n_rows;
    uint32_t pitch, filter_pitch, filter_col, n_constraints, n_challenges, kind, param;
    // FILTER_COLUMN: filter(row) = column filter_col.  FILTER_SELECTOR: `filter` is the constants/sigmas leaf matrix, column filter_col the
    // gate's selector s, and filter(row) = selector_filter(s, gate_index, group_start, group_end, many_selectors); the gate constants are
    // its columns [const_col0, ...)
    uint32_t filter_mode, gate_index, group_start, group_end, many_selectors, const_col0;
    PiHash pi;
};

// acc[k][row] += filter(row) * sum_i powers[k][i] * constraint_i(row); POSEIDON: the instance of GATE_POSEIDON, else every other kind
template <int NCH, bool POSEIDON = false>
__global__ void __launch_bounds__(128) gate_quotient_kernel(const QuotientArgs a) {
    extern __shared__ uint64_t pw[];   // [NCH][n_constraints]
    for (uint32_t i = threadIdx.x; i < NCH * a.n_constraints; i += blockDim.x) pw[i] = a.powers[i];
    __syncthreads();
    const uint64_t row = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= a.n_rows) return;
    const uint64_t* r = a.rows + row * a.pitch;
    uint64_t acc[NCH];
#pragma unroll
    for (int k = 0; k < NCH; k++) acc[k] = 0;
    uint32_t i = 0;
    auto wires = [&](int j) { return gl::canon(__ldg(r + j)); };
    auto emit = [&](uint64_t v) {
#pragma unroll
        for (int k = 0; k < NCH; k++) acc[k] = gl::add(acc[k], gl::mulc(v, pw[k * a.n_constraints + i]));
        i++;
    };
    if constexpr (POSEIDON)
        poseidon_gate(wires, emit);
    else
        eval_gate((int)a.kind, a.param, wires, [&](int j) { return gl::canon(__ldg(a.filter + row * a.filter_pitch + a.const_col0 + j)); },
                  a.pi.w, emit);
    uint64_t f = 1;
    if (a.filter_mode != FILTER_NONE) {
        f = gl::canon(__ldg(a.filter + row * a.filter_pitch + a.filter_col));
        if (a.filter_mode == FILTER_SELECTOR) f = selector_filter(f, a.gate_index, a.group_start, a.group_end, a.many_selectors);
    }
#pragma unroll
    for (int k = 0; k < NCH; k++) {
        uint64_t v = a.filter_mode != FILTER_NONE ? gl::mulc(acc[k], f) : acc[k];
        uint64_t* dst = a.acc + (uint64_t)k * a.n_rows + row;
        *dst = gl::add(*dst, v);
    }
}

// tail of compute_quotient_polys: vals[i][k] = acc[k][bitrev(i)] / Z_H(g w_R^i), natural point order, row-major [R][pitch];
// Z_H on the coset takes 2^rate_bits values: zh_inv[i mod 2^rate_bits] (plonky2 plonk/plonk_common.rs · ZeroPolyOnCoset::eval_inverse)
__global__ void quotient_gather_kernel(const uint64_t* __restrict__ acc, uint64_t* __restrict__ out, uint32_t pitch, uint32_t n_ch, uint32_t bits,
                                       uint32_t rate_bits, const uint64_t* __restrict__ zh_inv) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x, R = 1ULL << bits;
    if (i >= R) return;
    const uint64_t src = gl::bitrev32((uint32_t)i, bits);
    const uint64_t zi = zh_inv[i & ((1u << rate_bits) - 1)];
    for (uint32_t k = 0; k < pitch; k++) out[i * pitch + k] = k < n_ch ? gl::mulc(acc[(uint64_t)k * R + src], zi) : 0;
}
// coefficients of the coset iFFT -> the quotient chunk polynomials: out[(k * n_chunks + c)][m] = coeffs[c * N + m][k] * shift^-(c N + m)
__global__ void quotient_chunks_kernel(const uint64_t* __restrict__ coeffs, uint32_t pitch, uint32_t n_ch, uint32_t log_n, uint32_t rate_bits,
                                       const uint64_t* __restrict__ shift_inv_pow, uint64_t* __restrict__ out) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x, R = 1ULL << (log_n + rate_bits), N = 1ULL << log_n;
    if (j >= R) return;
    const uint64_t c = j >> log_n, m = j & (N - 1), s = shift_inv_pow[j];
    for (uint32_t k = 0; k < n_ch; k++) out[((uint64_t)k << rate_bits | c) * N + m] = gl::mulc(coeffs[j * pitch + k], s);
}

// Poseidon2Generator::run_once for a batch of rows: in[n][13] = 12 inputs + swap flag -> out[n][out_pitch] (135 wires)
__global__ void poseidon2_witness_kernel(const uint64_t* __restrict__ in, uint64_t n, uint64_t* __restrict__ out, uint32_t out_pitch) {
    const uint64_t row = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= n) return;
    const uint64_t* x = in + row * 13;
    uint64_t* w = out + row * out_pitch;
    uint64_t s[P2_WIDTH];
#pragma unroll
    for (int i = 0; i < P2_WIDTH; i++) { s[i] = gl::canon(x[i]); w[i] = s[i]; }
    const uint64_t swap = gl::canon(x[12]);
    w[P2_WIRE_SWAP] = swap;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        w[P2_START_DELTA + i] = gl::mulc(swap, gl::sub(s[i + 4], s[i]));
        if (swap == 1) { const uint64_t t = s[i]; s[i] = s[i + 4]; s[i + 4] = t; }   // `if swap_value == F::ONE { state.swap(i, 4 + i) }`
    }
    matmul_external(s);
#pragma unroll 1
    for (int r = 0; r < P2_RF_BEGIN; r++) {
#pragma unroll
        for (int i = 0; i < P2_WIDTH; i++) {
            const uint64_t v = gl::add(s[i], poseidon2::RC[r][i]);
            if (r != 0) w[P2_START_RF_BEGIN + P2_WIDTH * (r - 1) + i] = v;
            s[i] = sbox7(v);
        }
        matmul_external(s);
    }
#pragma unroll 1
    for (int r = 0; r < P2_RP; r++) {
        const uint64_t v = gl::add(s[0], poseidon2::RC_MID[r]);
        w[P2_START_PARTIAL + r] = v;
        s[0] = sbox7(v);
        matmul_internal(s);
    }
#pragma unroll 1
    for (int r = P2_RF_BEGIN; r < P2_RF_END; r++) {
#pragma unroll
        for (int i = 0; i < P2_WIDTH; i++) {
            const uint64_t v = gl::add(s[i], poseidon2::RC[r][i]);
            w[P2_START_RF_END + P2_WIDTH * (r - P2_RF_BEGIN) + i] = v;
            s[i] = sbox7(v);
        }
        matmul_external(s);
    }
#pragma unroll
    for (int i = 0; i < P2_WIDTH; i++) w[P2_WIDTH + i] = s[i];
}

// PoseidonGenerator::run_once (gates/poseidon.rs) for a batch of rows, poseidon2_witness_kernel's shape: in[n][13] -> out[n][out_pitch]
__global__ void poseidon_witness_kernel(const uint64_t* __restrict__ in, uint64_t n, uint64_t* __restrict__ out, uint32_t out_pitch) {
    const uint64_t row = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= n) return;
    const uint64_t* x = in + row * 13;
    uint64_t* w = out + row * out_pitch;
    uint64_t s[P2_WIDTH];
#pragma unroll
    for (int i = 0; i < P2_WIDTH; i++) { s[i] = gl::canon(x[i]); w[i] = s[i]; }
    const uint64_t swap = gl::canon(x[12]);
    w[P2_WIRE_SWAP] = swap;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        w[P2_START_DELTA + i] = gl::mulc(swap, gl::sub(s[i + 4], s[i]));
        if (swap == 1) { const uint64_t t = s[i]; s[i] = s[i + 4]; s[i + 4] = t; }   // `if swap_value == F::ONE { state.swap(i, 4 + i) }`
    }
    poseidon_rounds(s, [&](int wire, uint64_t v) {
        w[wire] = v;
        return v;
    });
#pragma unroll
    for (int i = 0; i < P2_WIDTH; i++) w[P2_WIDTH + i] = s[i];
}

}  // namespace gates
