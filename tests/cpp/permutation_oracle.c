/*
 * TEST INFRASTRUCTURE — the permutation argument and the tail of compute_quotient_polys restated in C (+ OpenMP), to check the device
 * at prover sizes where the Python big-integer restatements of oracle/gates_oracle.py are too slow.  Loaded by
 * tests/permutation_oracle.py, which builds it into a temporary directory keyed by the source's hash, so a read-only tree works.
 * Field arithmetic as oracle/gl_oracle.c (goldilocks_field.rs · reduce128).
 */
#include <stdint.h>
#include <stdlib.h>
#ifdef _OPENMP
#include <omp.h>
#endif

typedef unsigned __int128 u128;
#define GL_P 0xFFFFFFFF00000001ULL
#define GL_EPS 0xFFFFFFFFULL

static inline uint64_t gl_canon(uint64_t x) { return x >= GL_P ? x - GL_P : x; }
static inline uint64_t gl_add(uint64_t a, uint64_t b)
{ /* a, b canonical */
    uint64_t s = a + b;
    uint64_t over = (uint64_t)0 - (uint64_t)((s < a) | (s >= GL_P));
    return s - (GL_P & over);
}
static inline uint64_t gl_sub(uint64_t a, uint64_t b)
{
    uint64_t d = a - b;
    return d + (GL_P & ((uint64_t)0 - (uint64_t)(a < b)));
}
static inline uint64_t gl_reduce128(u128 x)
{ /* 2^64 = 2^32 - 1, 2^96 = -1 (mod p); returns canonical */
    uint64_t lo = (uint64_t)x, hi = (uint64_t)(x >> 64);
    uint64_t hh = hi >> 32, hl = hi & GL_EPS;
    uint64_t t0 = lo - hh;
    t0 -= GL_EPS & ((uint64_t)0 - (uint64_t)(lo < hh));
    uint64_t t1 = hl * GL_EPS;
    uint64_t t2 = t0 + t1;
    t2 += GL_EPS & ((uint64_t)0 - (uint64_t)(t2 < t0));
    return t2 - (GL_P & ((uint64_t)0 - (uint64_t)(t2 >= GL_P)));
}
static inline uint64_t gl_mul(uint64_t a, uint64_t b) { return gl_reduce128((u128)a * b); }
static uint64_t gl_pow(uint64_t b, uint64_t e)
{
    uint64_t r = 1;
    while (e) {
        if (e & 1) r = gl_mul(r, b);
        b = gl_mul(b, b);
        e >>= 1;
    }
    return r;
}
static uint64_t gl_inv(uint64_t a) { return gl_pow(a, GL_P - 2); }
static uint64_t gl_root_of_unity(unsigned n_log) { return gl_pow(1753635133440165772ULL, 1ULL << (32 - n_log)); }
static inline uint64_t bitrev64(uint64_t x, unsigned bits)
{
    uint64_t r = 0;
    for (unsigned i = 0; i < bits; i++) { r = (r << 1) | (x & 1); x >>= 1; }
    return r;
}

/* inverse DFT on the subgroup of order 2^log_n, natural order in and out: a[m] <- (1/n) sum_j a[j] w^-jm (radix-2 DIT with w^-1) */
static void ifft(uint64_t* a, unsigned log_n)
{
    const uint64_t n = 1ULL << log_n;
    for (uint64_t i = 0; i < n; i++) {
        const uint64_t j = bitrev64(i, log_n);
        if (i < j) { const uint64_t t = a[i]; a[i] = a[j]; a[j] = t; }
    }
    for (unsigned s = 1; s <= log_n; s++) {
        const uint64_t m = 1ULL << s, half = m >> 1, w_m = gl_inv(gl_root_of_unity(s));
#pragma omp parallel for schedule(static)
        for (int64_t k = 0; k < (int64_t)n; k += (int64_t)m) {
            uint64_t w = 1;
            for (uint64_t j = 0; j < half; j++) {
                const uint64_t u = a[k + j], t = gl_mul(w, a[k + j + half]);
                a[k + j] = gl_add(u, t);
                a[k + j + half] = gl_sub(u, t);
                w = gl_mul(w, w_m);
            }
        }
    }
    const uint64_t n_inv = gl_inv(n % GL_P);
    for (uint64_t i = 0; i < n; i++) a[i] = gl_mul(a[i], n_inv);
}

/* ---- permutation argument (plonky2 plonk/prover.rs · wires_permutation_partial_products_and_zs, plonk/vanishing_poly.rs ·
 * eval_vanishing_poly_base_batch, plonk/prover.rs · compute_quotient_polys' tail).  Restated from the published definitions, one
 * row at a time: every denominator product is inverted on its own with a Fermat power (no batch inverse), L_0 and Z_H are computed
 * from x with powers (no per-coset tables).  Every input word may be non-canonical. ---- */

/* wires, sigmas: [n_routed][n] values on the subgroup (natural order, column-major); k_is [n_routed]; betas, gammas [n_ch].
 * out: [n_ch * n_chunks][n] in prove()'s order: Z of every challenge, then each challenge's n_chunks - 1 partial products.
 * With q_ic = prod_{j in chunk c} (w_ij + beta k_j x_i + gamma) / (w_ij + beta sigma_ij + gamma), the running product over (i, c) in
 * row-major order starts at Z(x_0) = 1; pp_c(x_i) is the product after chunk c of row i, and the product after row i is Z(x_{i+1}). */
int glo_partial_products(const uint64_t* wires, const uint64_t* sigmas, uint32_t n_routed, uint32_t log_n, const uint64_t* k_is,
                         const uint64_t* betas, const uint64_t* gammas, uint32_t n_ch, uint32_t degree, uint64_t* out)
{
    if (n_routed == 0 || degree == 0 || n_ch == 0 || log_n > 32) return -1;
    const uint64_t n = 1ULL << log_n;
    const uint32_t n_chunks = (n_routed + degree - 1) / degree, n_pp = n_chunks - 1;
    const uint64_t w = gl_root_of_unity(log_n);
    uint64_t* q = (uint64_t*)malloc(sizeof(uint64_t) * n * n_chunks);
    if (!q) return -1;
    for (uint32_t k = 0; k < n_ch; k++) {
        const uint64_t beta = gl_canon(betas[k]), gamma = gl_canon(gammas[k]);
#pragma omp parallel for schedule(static)
        for (int64_t i = 0; i < (int64_t)n; i++) {
            const uint64_t x = gl_pow(w, (uint64_t)i);
            for (uint32_t c = 0; c < n_chunks; c++) {
                uint64_t pn = 1, pd = 1;
                for (uint32_t j = c * degree; j < n_routed && j < (c + 1) * degree; j++) {
                    const uint64_t wv = gl_canon(wires[(uint64_t)j * n + i]);
                    pn = gl_mul(pn, gl_add(gl_add(wv, gl_mul(gl_mul(beta, gl_canon(k_is[j])), x)), gamma));
                    pd = gl_mul(pd, gl_add(gl_add(wv, gl_mul(beta, gl_canon(sigmas[(uint64_t)j * n + i]))), gamma));
                }
                q[(uint64_t)i * n_chunks + c] = gl_mul(pn, gl_inv(pd));
            }
        }
        uint64_t acc = 1;
        for (uint64_t i = 0; i < n; i++) {
            out[(uint64_t)k * n + i] = acc;
            for (uint32_t c = 0; c < n_chunks; c++) {
                acc = gl_mul(acc, q[i * n_chunks + c]);
                if (c < n_pp) out[((uint64_t)n_ch + (uint64_t)k * n_pp + c) * n + i] = acc;
            }
        }
    }
    free(q);
    return 0;
}

/* The permutation part of the vanishing terms at LDE leaf rows, alpha-reduced.  Leaf row `row` of a rate-r commit of degree N = 2^log_n
 * is the coset point x = 7 w_R^bitrev(row) (R = N 2^r); Z(g x) sits at the row whose point index is bitrev(row) + 2^r (mod R).
 *   wires [R][wires_pitch] (routed wires at columns [0, n_routed)), sigmas [R][sigmas_pitch] (at [sigma_col0, sigma_col0 + n_routed)),
 *   zs [R][zs_pitch] (Z of every challenge, then each challenge's partial products); rows [n_rows]; out [n_rows][n_ch]:
 *   out[i][k] = sum_t alpha_k^t term_t(rows[i]) over terms = [L_0(x)(Z_c(x) - 1) for every c] ++ [check_partial_products of every c]. */
int glo_vanishing_permutation(const uint64_t* wires, uint32_t wires_pitch, const uint64_t* sigmas, uint32_t sigmas_pitch, uint32_t sigma_col0,
                              const uint64_t* zs, uint32_t zs_pitch, uint32_t log_n, uint32_t rate_bits, uint32_t n_routed, uint32_t degree,
                              const uint64_t* k_is, const uint64_t* betas, const uint64_t* gammas, const uint64_t* alphas, uint32_t n_ch,
                              const uint64_t* rows, uint64_t n_rows, uint64_t* out)
{
    if (n_routed == 0 || degree == 0 || n_ch == 0 || log_n + rate_bits > 32) return -1;
    const uint32_t bits = log_n + rate_bits, n_chunks = (n_routed + degree - 1) / degree, n_pp = n_chunks - 1;
    const uint32_t n_terms = n_ch * (1 + n_chunks);
    const uint64_t R = 1ULL << bits, n = 1ULL << log_n, w_r = gl_root_of_unity(bits);
    for (uint64_t i = 0; i < n_rows; i++)
        if (rows[i] >= R) return -1;
    const uint64_t n_inv = gl_inv(n % GL_P);
    int rc = 0;
#pragma omp parallel
    {
        uint64_t* terms = (uint64_t*)malloc(sizeof(uint64_t) * n_terms);
        if (!terms) {
#pragma omp atomic write
            rc = -1;
        }
#pragma omp for schedule(static)
        for (int64_t ii = 0; ii < (int64_t)n_rows; ii++) {
            if (!terms) continue;
            const uint64_t row = rows[ii], idx = bitrev64(row, bits);
            const uint64_t row_next = bitrev64((idx + (1ULL << rate_bits)) & (R - 1), bits);
            const uint64_t x = gl_mul(7, gl_pow(w_r, idx));
            const uint64_t l0 = gl_mul(gl_mul(gl_sub(gl_pow(x, n), 1), n_inv), gl_inv(gl_sub(x, 1)));
            const uint64_t* wr = wires + row * wires_pitch;
            const uint64_t* sr = sigmas + row * sigmas_pitch + sigma_col0;
            const uint64_t* zr = zs + row * zs_pitch;
            const uint64_t* zn = zs + row_next * zs_pitch;
            for (uint32_t c = 0; c < n_ch; c++) {
                const uint64_t beta = gl_canon(betas[c]), gamma = gl_canon(gammas[c]);
                const uint64_t z_x = gl_canon(zr[c]), z_gx = gl_canon(zn[c]);
                terms[c] = gl_mul(l0, gl_sub(z_x, 1));
                for (uint32_t ch = 0; ch < n_chunks; ch++) {
                    uint64_t pn = 1, pd = 1;
                    for (uint32_t j = ch * degree; j < n_routed && j < (ch + 1) * degree; j++) {
                        const uint64_t wv = gl_canon(wr[j]);
                        pn = gl_mul(pn, gl_add(gl_add(wv, gl_mul(gl_mul(beta, gl_canon(k_is[j])), x)), gamma));
                        pd = gl_mul(pd, gl_add(gl_add(wv, gl_mul(beta, gl_canon(sr[j]))), gamma));
                    }
                    const uint64_t prev = ch == 0 ? z_x : gl_canon(zr[n_ch + c * n_pp + ch - 1]);
                    const uint64_t next = ch + 1 < n_chunks ? gl_canon(zr[n_ch + c * n_pp + ch]) : z_gx;
                    terms[n_ch + c * n_chunks + ch] = gl_sub(gl_mul(prev, pn), gl_mul(next, pd));
                }
            }
            for (uint32_t k = 0; k < n_ch; k++) {   /* reduce_with_powers: Horner from the last term */
                const uint64_t alpha = gl_canon(alphas[k]);
                uint64_t acc = 0;
                for (uint32_t t = n_terms; t-- > 0;) acc = gl_add(gl_mul(acc, alpha), terms[t]);
                out[(uint64_t)ii * n_ch + k] = acc;
            }
        }
        free(terms);
    }
    return rc;
}

/* compute_quotient_polys' tail: acc [n_ch][R] in leaf order (row i = point bitrev(i)) holds the alpha-combined vanishing terms on the
 * coset 7 w_R^j.  quotient_j = acc(point j) / Z_H(7 w_R^j) with Z_H(x) = x^N - 1, then coset_ifft with shift 7 (ifft, then coefficient
 * m times 7^-m), split into 2^r chunks of N coefficients: out [(n_ch << r)][N], chunk c of challenge k at row (k << r) + c. */
int glo_quotient_chunks(const uint64_t* acc, uint32_t n_ch, uint32_t log_n, uint32_t rate_bits, uint64_t* out)
{
    const uint32_t bits = log_n + rate_bits;
    if (bits > 32) return -1;
    const uint64_t R = 1ULL << bits, n = 1ULL << log_n, w_r = gl_root_of_unity(bits), inv7 = gl_inv(7);
    uint64_t* zh_inv = (uint64_t*)malloc(sizeof(uint64_t) * R);
    uint64_t* vals = (uint64_t*)malloc(sizeof(uint64_t) * R);
    if (!zh_inv || !vals) { free(zh_inv); free(vals); return -1; }
#pragma omp parallel for schedule(static)
    for (int64_t j = 0; j < (int64_t)R; j++)
        zh_inv[j] = gl_inv(gl_sub(gl_pow(gl_mul(7, gl_pow(w_r, (uint64_t)j)), n), 1));
    for (uint32_t k = 0; k < n_ch; k++) {
        const uint64_t* a = acc + (uint64_t)k * R;
#pragma omp parallel for schedule(static)
        for (int64_t j = 0; j < (int64_t)R; j++) vals[j] = gl_mul(gl_canon(a[bitrev64((uint64_t)j, bits)]), zh_inv[j]);
        ifft(vals, bits);
        uint64_t s = 1;
        for (uint64_t m = 0; m < R; m++) {
            out[((uint64_t)k << rate_bits) * n + m] = gl_mul(vals[m], s);   /* chunk m / N of challenge k, coefficient m mod N */
            s = gl_mul(s, inv7);
        }
    }
    free(zh_inv);
    free(vals);
    return 0;
}

