/*
 * TEST INFRASTRUCTURE — the host side of OpeningSet::new's eval_commitment (plonky2 plonk/proof.rs): p.to_extension().eval(point) for
 * every polynomial of a batch, Horner from the top coefficient in F_p[X]/(X^2 - 7), one polynomial per OpenMP iteration.
 * Loaded by tests/opening_set_oracle.py and linked into the ABI test double's gl_batch_eval (tests/cpp/abi_test_double_batch_eval.cpp).
 * Field arithmetic as oracle/gl_oracle.c (goldilocks_field.rs · reduce128).
 */
#include <stdint.h>
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

/* polys: [n_polys][n] base-field coefficients (any 64-bit words); point: extension element (any words); out: [n_polys][2], canonical */
void glo_eval_ext(const uint64_t* polys, uint32_t n_polys, uint64_t n, const uint64_t point[2], uint64_t* out)
{
    const uint64_t z0 = gl_canon(point[0]), z1 = gl_canon(point[1]);
#pragma omp parallel for schedule(dynamic, 1)
    for (int64_t j = 0; j < (int64_t)n_polys; j++) {
        const uint64_t* f = polys + (uint64_t)j * n;
        uint64_t a0 = 0, a1 = 0;
        for (uint64_t k = n; k-- > 0;) {   /* acc = acc * z + f[k] */
            const uint64_t m0 = gl_add(gl_mul(a0, z0), gl_mul(7, gl_mul(a1, z1)));
            const uint64_t m1 = gl_add(gl_mul(a0, z1), gl_mul(a1, z0));
            a0 = gl_add(m0, gl_canon(f[k]));
            a1 = m1;
        }
        out[2 * j] = a0; out[2 * j + 1] = a1;
    }
}

int glo_eval_ext_threads(void)
{
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}
