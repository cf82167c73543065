// K6: FRI commit-phase helpers over the quadratic extension F_p[X]/(X^2 - 7).
//
// Replaces the arithmetic of plonky2 fri/src/prover.rs · fri_committed_trees (reverse_index_bits_in_place,
// chunk-by-arity flatten, reduce_with_powers fold) — semantics SURVEY.md A.7; the extension is the same W = 7
// binomial extension the reference uses in-circuit (/root/reference/src/p3/extension.rs:147-151,458-470).
// An extension element is two consecutive words [a0, a1]; an extension array is therefore a row-major matrix
// with 2 columns, which lets the coset NTT of the folded polynomial reuse ntt_pass_kernel<2>.
#pragma once
#include "gl_field.cuh"

namespace fri {

// dst[i] = canon(src[bitrev_bits(i)]) for extension elements (16 B each)
__global__ void bitrev_gather_ext_kernel(const ulonglong2* __restrict__ src, ulonglong2* __restrict__ dst, uint32_t bits) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (1u << bits)) return;
    ulonglong2 v = src[gl::bitrev32(i, bits)];
    dst[i] = make_ulonglong2(gl::canon(v.x), gl::canon(v.y));
}

__global__ void canon_kernel(uint64_t* __restrict__ a, uint64_t n) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) a[i] = gl::canon(a[i]);
}

// out[m] = sum_{t < arity} in[arity*m + t] * beta^t      (reduce_with_powers, Horner from the top)
__global__ void fold_kernel(const ulonglong2* __restrict__ in, ulonglong2* __restrict__ out, uint32_t n_out,
                            uint32_t arity, uint64_t beta0, uint64_t beta1) {
    uint32_t m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= n_out) return;
    gl::Ext beta = {beta0, beta1};
    gl::Ext acc = {0, 0};
    for (uint32_t t = arity; t-- > 0;) {
        ulonglong2 c = in[(size_t)arity * m + t];
        acc = gl::ext_mul(acc, beta);
        acc.a0 = gl::add(acc.a0, c.x);
        acc.a1 = gl::add(acc.a1, c.y);
    }
    out[m] = make_ulonglong2(acc.a0, acc.a1);
}

}  // namespace fri
