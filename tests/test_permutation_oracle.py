"""CPU: the C restatements of the permutation argument and the quotient tail (tests/cpp/permutation_oracle.c), which check the device
at prover sizes in tests/test_permutation_quotient_gpu.py, against the Python big-integer restatements.  No GPU needed."""
import numpy as np
import pytest

import gates_oracle as go
import gl_oracle as o
import permutation_oracle as po
from oracle_c import P


def _noncanonical(rng, shape):
    """field elements as u64 words, a quarter of them in the non-canonical form v + p (v < 2^32 - 1)"""
    a = rng.integers(0, P, size=shape, dtype=np.uint64)
    small = rng.integers(0, 2**32 - 1, size=shape, dtype=np.uint64)
    return np.where(rng.random(shape) < 0.25, small + np.uint64(P), a)


@pytest.mark.parametrize("log_n,n_routed,degree,n_ch", [(0, 5, 2, 1), (2, 7, 3, 2), (3, 9, 1, 3), (3, 13, 4, 4), (4, 6, 6, 2)])
def test_permutation_oracle_c_matches_python(log_n, n_routed, degree, n_ch):
    """the C restatements of tests/cpp/permutation_oracle.c (glo_partial_products, glo_vanishing_permutation, glo_quotient_chunks), which
    check the device at prover sizes, against the Python big-integer restatements of oracle/gates_oracle.py on small instances: every
    challenge count, an uneven last chunk, degree 1, non-canonical words in every input"""
    rng = np.random.default_rng(1000 * log_n + 10 * n_routed + n_ch)
    n = 1 << log_n
    wires, sigmas = _noncanonical(rng, (n_routed, n)), _noncanonical(rng, (n_routed, n))
    k_is, betas, gammas, alphas = (_noncanonical(rng, m) for m in (n_routed, n_ch, n_ch, n_ch))
    ints = lambda a: [int(v) for v in np.asarray(a).reshape(-1)]
    got = po.partial_products(wires, sigmas, k_is, betas, gammas, degree)
    want = go.partial_products_and_zs([ints(c) for c in wires], [ints(c) for c in sigmas], ints(k_is), ints(betas), ints(gammas), degree, log_n)
    assert got.tolist() == want
    # vanishing terms at every leaf row of random rate-r leaf matrices (the terms are defined for any values)
    n_chunks = -(-n_routed // degree)
    for r in (0, 1, 3):
        bits, R = log_n + r, n << r
        lw, ls, lz = _noncanonical(rng, (R, n_routed + 2)), _noncanonical(rng, (R, n_routed + 5)), _noncanonical(rng, (R, n_ch * n_chunks))
        got = po.vanishing_permutation(lw, ls, 3, lz, np.arange(R), log_n, r, n_routed, degree, k_is, betas, gammas, alphas)
        w_R = o.primitive_root_of_unity(bits)
        for row in range(R):
            idx = int(format(row, "0%db" % bits)[::-1] or "0", 2)
            nxt = (idx + (1 << r)) % R
            row_next = int(format(nxt, "0%db" % bits)[::-1] or "0", 2)
            x = 7 * pow(w_R, idx, P) % P
            terms = go.vanishing_permutation_terms(ints(lw[row, :n_routed]), ints(ls[row, 3:3 + n_routed]), ints(lz[row]), ints(lz[row_next]),
                                                   x, ints(k_is), ints(betas), ints(gammas), degree, log_n)
            assert got[row].tolist() == [go.reduce_with_powers(terms, int(a) % P) for a in alphas], (r, row)
    # the quotient tail against a naive inverse DFT on the coset
    r = 2
    bits, R = log_n + r, n << r
    acc = _noncanonical(rng, (n_ch, R))
    got = po.quotient_chunks(acc, log_n, r)
    w_R = o.primitive_root_of_unity(bits)
    for k in range(n_ch):
        pts = [7 * pow(w_R, j, P) % P for j in range(R)]
        vals = [int(acc[k, int(format(j, "0%db" % bits)[::-1], 2)]) * pow(pow(x, n, P) - 1, P - 2, P) % P for j, x in enumerate(pts)]
        # coefficient m of q with q(7 w^j) = vals[j]: (1/R) 7^-m sum_j vals[j] w^-jm
        coeffs = [pow(R, P - 2, P) * pow(7, (P - 2) * m, P) * sum(v * pow(w_R, (R - j * m % R) % R, P) for j, v in enumerate(vals)) % P
                  for m in range(R)]
        assert got[k << r:(k + 1) << r].reshape(-1).tolist() == coeffs, k
