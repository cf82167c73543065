// K9: front half of PolynomialBatch::prove_openings (plonky2 fri/oracle.rs) on device-resident coefficient matrices:
//   composition  F = sum_j alpha^j f_j            (util/reducing.rs · ReducingFactor::reduce_polys_base)
//   quotient     (F(X) - F(z)) / (X - z)          (field/polynomial/division.rs · divide_by_linear, padded back to N)
//   final_poly <- final_poly * alpha^count + quotient   (ReducingFactor::shift_poly, then +=)
// driven in the reference from /root/reference/src/p3/mod.rs:260 (`data.prove`).  Polynomials are columns of the
// row-major coefficient matrices [N][pitch] the commits left in HBM, so coefficient k of every polynomial of a batch is
// one contiguous run of a row — the same access pattern as the leaf hash.  All arithmetic is exact field arithmetic, so
// any association order gives the reference's canonical result.
#pragma once
#include "fri.cuh"

namespace openings {

struct PolyRef {
    const uint64_t* base;   // coefficient matrix of the oracle
    uint32_t pitch, col;
};

// out[k] = sum_j pw[j] * f_j[k]  (pw[j] = alpha^j, extension; f_j base field).  One thread per coefficient index.
__global__ void reduce_polys_base_kernel(const PolyRef* __restrict__ polys, const ulonglong2* __restrict__ pw, uint32_t n_polys,
                                         uint32_t n, ulonglong2* __restrict__ out) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    uint64_t a0 = 0, a1 = 0;
    for (uint32_t j = 0; j < n_polys; j++) {
        const PolyRef r = polys[j];
        const uint64_t v = r.base[(size_t)k * r.pitch + r.col];
        const ulonglong2 w = pw[j];
        a0 = gl::add(a0, gl::mulc(v, w.x));
        a1 = gl::add(a1, gl::mulc(v, w.y));
    }
    out[k] = make_ulonglong2(a0, a1);
}

__device__ __forceinline__ fri::Ext ext_add(fri::Ext a, fri::Ext b) { return {gl::add(a.a0, b.a0), gl::add(a.a1, b.a1)}; }

// In place: f (n extension coefficients) -> q with q[k] = f[k+1] + z*q[k+1], q[n-1] = 0  (synthetic division by X - z).
// One CTA; thread t owns the chunk [t*L, (t+1)*L): (1) Horner value of its chunk, (2) a serial right-to-left carry over
// the <= 1024 chunk values by thread 0, (3) the chunk's quotient coefficients from its carry-in.
__global__ void divide_by_linear_kernel(ulonglong2* __restrict__ f, uint32_t n, uint64_t z0, uint64_t z1) {
    __shared__ fri::Ext chunk_val[1024];
    __shared__ fri::Ext carry_in[1024];
    const uint32_t T = blockDim.x, t = threadIdx.x, L = n / T;   // n, T powers of two, T <= n
    const fri::Ext z = {z0, z1};
    // (1) h_t = sum_{i in chunk} f[i] z^(i - t*L)
    fri::Ext h = {0, 0};
    for (uint32_t i = L; i-- > 0;) {
        const ulonglong2 c = f[(size_t)t * L + i];
        h = fri::ext_mul(h, z);
        h = ext_add(h, {c.x, c.y});
    }
    chunk_val[t] = h;
    __syncthreads();
    // (2) carry_in[t] = sum_{i >= (t+1)L} f[i] z^(i - (t+1)L)  (= q[(t+1)L - 1], the quotient coefficient just left of chunk t+1)
    if (t == 0) {
        fri::Ext zL = {1, 0};
        for (uint32_t i = 0; i < L; i++) zL = fri::ext_mul(zL, z);
        fri::Ext acc = {0, 0};
        for (uint32_t u = T; u-- > 0;) {
            carry_in[u] = acc;
            acc = ext_add(fri::ext_mul(acc, zL), chunk_val[u]);
        }
    }
    __syncthreads();
    // (3) q[k] = f[k+1] + z*q[k+1] inside the chunk, starting from q[(t+1)L - 1] = carry_in[t]
    fri::Ext q = carry_in[t];
    for (uint32_t i = L; i-- > 0;) {
        const size_t k = (size_t)t * L + i;
        const ulonglong2 c = f[k];                      // f[k] is needed for q[k-1]; read before overwriting
        f[k] = make_ulonglong2(q.a0, q.a1);
        q = ext_add(fri::ext_mul(q, z), {c.x, c.y});
    }
}

// final[k] = final[k] * s + q[k]
__global__ void shift_add_kernel(ulonglong2* __restrict__ fin, const ulonglong2* __restrict__ q, uint32_t n, uint64_t s0, uint64_t s1) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const ulonglong2 a = fin[k], b = q[k];
    fri::Ext r = fri::ext_mul({a.x, a.y}, {s0, s1});
    fin[k] = make_ulonglong2(gl::add(r.a0, b.x), gl::add(r.a1, b.y));
}

// ---- OpeningSet::new (plonky2 plonk/proof.rs, the eval_commitment closure) ----------------------------------------------------------
// out[p][j] = sum_{k<N} coeffs[k][j] * z_p^k for every live column j of one resident [N][pitch] coefficient matrix, 1 or 2 points.
// Stage 1 (batch_eval_partial_kernel): CTA (x, y) owns rows [x * subs * sub_rows, (x + 1) * subs * sub_rows) of the column tile
// [y * wc, (y + 1) * wc).  Its threads are `lanes` row lanes of `wc` consecutive columns, so a warp reads consecutive words of one or two
// rows, and the matrix is read once whatever the number of points.  The powers z_p^k of a sub-chunk's rows sit in shared memory: the
// first sub-chunk's by square-and-multiply over the host's z_p^(2^b), each later one by one product with z_p^sub_rows, so an element
// costs one base x extension product per point (2 mulc + 2 add).  The lanes are summed in shared memory and the CTA writes
// partial[x][p][j].  Stage 2 (batch_eval_reduce_kernel) sums the partials over x.  No atomics: the arithmetic is exact, so any
// summation order gives the same canonical words.
constexpr uint32_t EVAL_SUB = 128;       // rows per shared-memory power tile
constexpr uint32_t EVAL_THREADS = 256;   // most threads of a stage-1 CTA
constexpr uint32_t EVAL_MAX_PARTS = 1024;
constexpr uint32_t EVAL_BATCH = 8;       // coefficient loads a thread issues before it multiplies

struct EvalPoints { uint64_t z2k[2][32][2]; };   // z_p^(2^b), canonical

__device__ __forceinline__ fri::Ext ext_pow_table(const uint64_t (*z2k)[2], uint64_t e) {
    fri::Ext r = {1, 0};
    for (uint32_t b = 0; e; b++, e >>= 1)
        if (e & 1) r = fri::ext_mul(r, {z2k[b][0], z2k[b][1]});
    return r;
}

template <int NP>
__global__ void __launch_bounds__(EVAL_THREADS) batch_eval_partial_kernel(const uint64_t* __restrict__ coeffs, uint32_t pitch,
                                                                          uint32_t leaf_len, uint32_t wc, uint32_t lanes, uint32_t sub_rows,
                                                                          uint32_t subs, const EvalPoints pts, ulonglong2* __restrict__ partial) {
    __shared__ fri::Ext pw[NP][EVAL_SUB];
    __shared__ fri::Ext red[NP][EVAL_THREADS];
    const uint32_t t = threadIdx.x, lane = t / wc, cl = t - lane * wc, col = blockIdx.y * wc + cl;
    const bool live = lane < lanes && col < leaf_len;
    const uint32_t log_sub = 31 - __clz(sub_rows);
    const uint64_t row0 = (uint64_t)blockIdx.x * subs * sub_rows;
    fri::Ext acc[NP];
#pragma unroll
    for (int p = 0; p < NP; p++) acc[p] = {0, 0};
    for (uint32_t s = 0; s < subs; s++) {
        const uint64_t r0 = row0 + (uint64_t)s * sub_rows;
        __syncthreads();   // every thread is done with the previous tile
        for (uint32_t i = t; i < sub_rows; i += blockDim.x) {
#pragma unroll
            for (int p = 0; p < NP; p++)
                pw[p][i] = s == 0 ? ext_pow_table(pts.z2k[p], r0 + i)
                                  : fri::ext_mul(pw[p][i], {pts.z2k[p][log_sub][0], pts.z2k[p][log_sub][1]});
        }
        __syncthreads();
        if (live) {
            const uint64_t* src = coeffs + r0 * pitch + col;
            for (uint32_t rb = lane; rb < sub_rows; rb += EVAL_BATCH * lanes) {
                uint64_t v[EVAL_BATCH];   // all loads of a batch are issued before any arithmetic: EVAL_BATCH reads in flight per thread
#pragma unroll
                for (uint32_t u = 0; u < EVAL_BATCH; u++) {
                    const uint32_t r = rb + u * lanes;
                    v[u] = r < sub_rows ? src[(uint64_t)r * pitch] : 0;
                }
#pragma unroll
                for (uint32_t u = 0; u < EVAL_BATCH; u++) {
                    const uint32_t r = rb + u * lanes;
                    if (r < sub_rows) {
#pragma unroll
                        for (int p = 0; p < NP; p++) {
                            const fri::Ext w = pw[p][r];
                            acc[p].a0 = gl::add(acc[p].a0, gl::mulc(v[u], w.a0));
                            acc[p].a1 = gl::add(acc[p].a1, gl::mulc(v[u], w.a1));
                        }
                    }
                }
            }
        }
    }
#pragma unroll
    for (int p = 0; p < NP; p++) red[p][t] = acc[p];
    __syncthreads();
    if (lane == 0 && col < leaf_len) {
#pragma unroll
        for (int p = 0; p < NP; p++) {
            fri::Ext sum = red[p][cl];
            for (uint32_t l = 1; l < lanes; l++) sum = ext_add(sum, red[p][l * wc + cl]);
            partial[((size_t)blockIdx.x * NP + p) * leaf_len + col] = make_ulonglong2(sum.a0, sum.a1);
        }
    }
}

// out[i] = sum_x partial[x][i], i < n_out (= n_points * leaf_len).  Block (32, 32): threadIdx.x walks i (coalesced), threadIdx.y walks x.
__global__ void batch_eval_reduce_kernel(const ulonglong2* __restrict__ partial, uint32_t n_parts, uint32_t n_out, ulonglong2* __restrict__ out) {
    __shared__ fri::Ext red[32][33];
    const uint32_t i = blockIdx.x * 32 + threadIdx.x;
    fri::Ext sum = {0, 0};
    if (i < n_out)
        for (uint32_t x = threadIdx.y; x < n_parts; x += 32) {
            const ulonglong2 v = partial[(size_t)x * n_out + i];
            sum = ext_add(sum, {v.x, v.y});
        }
    red[threadIdx.y][threadIdx.x] = sum;
    __syncthreads();
    if (threadIdx.y == 0 && i < n_out) {
        for (uint32_t y = 1; y < 32; y++) sum = ext_add(sum, red[y][threadIdx.x]);
        out[i] = make_ulonglong2(sum.a0, sum.a1);
    }
}

}  // namespace openings
