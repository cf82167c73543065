"""The permutation argument and the quotient commit on the device at prover sizes, against the C restatements of
tests/cpp/permutation_oracle.c (glo_partial_products, glo_vanishing_permutation, glo_quotient_chunks) and oracle/gl_oracle.c (glo_commit),
word for word:

- gl_partial_products up to 2^20 rows, so the running product's segmented scan runs with L = ceil(N / 1024) rows per thread from 1 to 1024,
  at every challenge count, up to MAX_CHUNKS chunks, an uneven last chunk and degree 1;
- gl_quotient_add_permutation at every challenge count 1..4 and every rate_bits 0..6, every row up to 2^16 LDE rows, and at the wrapper
  circuit's 2^19 rows every row whose "next" point wraps around the coset plus 4096 others;
- gl_quotient_commit at every challenge count against every rate_bits 0..6, down to N = 1;
- the verifier's identity at a random zeta on whole pipelines up to the wrapper's 2^16 x 80 routed wires, and its negative control.

Every host-side input (wires, sigmas, k_is, betas, gammas, alphas) carries non-canonical words v + p at many positions."""
import ctypes

import numpy as np
import pytest

import gates_oracle as go
import opening_set_oracle as oso
import permutation_oracle as po

P = go.P
GL_ERR_INVALID, GL_ERR_UNSUPPORTED = -1, -5
GENERATOR = 1753635133440165772          # 2^32-th root of unity
BASE_SUM = (13, 2 | 2 << 8)              # BaseSumGate<2> with 2 limbs: 3 wires, 3 constraints, no constants


def _field(rng, shape, frac=0.25):
    """random field elements as u64 words; about `frac` of them in the non-canonical form v + p (v < 2^32 - 1)"""
    a = rng.integers(0, P, size=shape, dtype=np.uint64)
    small = rng.integers(0, 2**32 - 1, size=shape, dtype=np.uint64)
    return np.where(rng.random(shape) < frac, small + np.uint64(P), a)


def _noncanonical_form(rng, a, frac=0.5):
    """the same field elements, with about `frac` of those that have a second u64 representation (v < 2^32 - 1) written as v + p"""
    a = np.asarray(a, dtype=np.uint64)
    return np.where((a < np.uint64(2**32 - 1)) & (rng.random(a.shape) < frac), a + np.uint64(P), a)


def _canon(a):
    a = np.asarray(a, dtype=np.uint64)
    return np.where(a >= np.uint64(P), a - np.uint64(P), a)


def _ints(a):
    return [int(v) % P for v in np.asarray(a).reshape(-1)]


def _bitrev(x, bits):
    x = np.asarray(x, dtype=np.uint64)
    r = np.zeros_like(x)
    for b in range(bits):
        r = (r << np.uint64(1)) | ((x >> np.uint64(b)) & np.uint64(1))
    return r


def _subgroup(log_n):
    w, xs, cur = pow(GENERATOR, 1 << (32 - log_n), P), [], 1
    for _ in range(1 << log_n):
        xs.append(cur)
        cur = cur * w % P
    return np.array(xs, dtype=np.uint64)


def _copy_permutation(rng, n_routed, log_n, k_is, cycle_len=5):
    """wires [n_routed][N] constant on the cycles of a random permutation sigma of the (column, row) cells, and the sigma polynomials'
    values sigma_j(x_i) = k_{j'} x_{i'} with (j', i') = sigma(j, i).  A quarter of the cycle values are small, and about half of the
    cells that hold a small value hold it in the non-canonical form v + p."""
    n = 1 << log_n
    cells = n_routed * n
    perm = rng.permutation(cells)
    t = np.arange(cells)
    start = t - t % cycle_len
    nxt = start + (t - start + 1) % np.minimum(cycle_len, cells - start)
    sigma = np.empty(cells, dtype=np.int64)
    sigma[perm] = perm[nxt]
    n_cycles = -(-cells // cycle_len)
    vals = np.where(rng.random(n_cycles) < 0.25, rng.integers(0, 2**32 - 1, size=n_cycles, dtype=np.uint64),
                    rng.integers(0, P, size=n_cycles, dtype=np.uint64))
    wires = np.empty(cells, dtype=np.uint64)
    wires[perm] = vals[t // cycle_len]
    ids = (np.asarray(_canon(k_is), dtype=object)[:, None] * _subgroup(log_n).astype(object)[None, :] % P).astype(np.uint64).reshape(-1)
    return _noncanonical_form(rng, wires).reshape(n_routed, n), ids[sigma].reshape(n_routed, n)


def _mod_sub(a, b):
    a, b = np.asarray(a, dtype=np.uint64), np.asarray(b, dtype=np.uint64)
    return np.where(a >= b, a - b, a + (np.uint64(P) - b))


# ------------------------------------------------------------------------------------------------ gl_partial_products
# (log_n, n_routed, degree, n_ch): N = 1; one chunk (no partial-product columns); N < 1024 (idle threads); L = 1 exactly; L = 2; 11 chunks
# with a one-wire last chunk; 16 chunks = MAX_CHUNKS; degree 1; the wrapper circuit's shape with a copy permutation; L = 1024
PP_CASES = [(0, 80, 8, 2), (1, 8, 8, 1), (9, 80, 8, 4), (10, 80, 8, 2), (11, 80, 8, 3), (12, 81, 8, 2), (13, 80, 5, 1), (14, 7, 1, 4),
            (16, 80, 8, 2), (20, 80, 8, 2)]


@pytest.mark.gpu
@pytest.mark.parametrize("log_n,n_routed,degree,n_ch", PP_CASES)
def test_partial_products_sweep(ctx, oc, log_n, n_routed, degree, n_ch):
    import plonky25_b200 as g
    rng = np.random.default_rng(7000 + 100 * log_n + n_routed)
    n = 1 << log_n
    betas, gammas = _field(rng, n_ch, 0.5), _field(rng, n_ch, 0.5)
    permuted = log_n == 16
    if permuted:
        k_is = _noncanonical_form(rng, [pow(7, j, P) for j in range(n_routed)])
        wires, sigmas = _copy_permutation(rng, n_routed, log_n, k_is)
    else:
        k_is = _field(rng, n_routed)
        wires, sigmas = _field(rng, (n_routed, n)), _field(rng, (n_routed, n))
    got = g.partial_products_and_zs(list(wires), list(sigmas), k_is, betas, gammas, degree, ctx=ctx)
    want = po.partial_products(wires, sigmas, k_is, betas, gammas, degree)
    assert got.shape == want.shape == (n_ch * -(-n_routed // degree), n)
    bad = np.argwhere(got != want)
    assert bad.size == 0, f"{len(bad)} words differ, first (column, row) {bad[:4].tolist()}"
    if permuted:
        # the argument closes: Z(x_0) = 1, and Z(x_{N-1}) times the last row's quotients returns to 1
        x_last = pow(GENERATOR, (n - 1) << (32 - log_n), P)
        w_last, s_last, k = _ints(wires[:, -1]), _ints(sigmas[:, -1]), _ints(k_is)
        for c, (beta, gamma) in enumerate(zip(_ints(betas), _ints(gammas))):
            assert int(got[c, 0]) == 1
            num = den = 1
            for j in range(n_routed):
                num = num * (w_last[j] + beta * k[j] % P * x_last + gamma) % P
                den = den * (w_last[j] + beta * s_last[j] + gamma) % P
            assert int(got[c, n - 1]) * num % P == den, "the running product does not close"


def _partial_products_rc(ctx, n_routed, log_n, n_ch, degree):
    n = 1 << log_n
    cols = [np.full(n, 3 + j, dtype=np.uint64) for j in range(n_routed)]
    ptrs = (ctypes.c_void_p * n_routed)(*[c.ctypes.data for c in cols])
    k = np.arange(1, n_routed + 1, dtype=np.uint64)
    bg = np.arange(5, 5 + max(n_ch, 1), dtype=np.uint64)
    out = np.zeros(max(n_ch, 1) * n_routed * n, dtype=np.uint64)
    return ctx.lib.gl_partial_products(ctx.handle, ptrs, ptrs, n_routed, log_n, k.ctypes.data, bg.ctypes.data, bg.ctypes.data, n_ch, degree,
                                       out.ctypes.data)


@pytest.mark.gpu
def test_partial_products_refusals(ctx):
    assert _partial_products_rc(ctx, 16, 3, 1, 1) == 0                       # MAX_CHUNKS = 16 chunks
    assert _partial_products_rc(ctx, 17, 3, 1, 1) == GL_ERR_UNSUPPORTED      # 17 chunks
    assert _partial_products_rc(ctx, 8, 3, 0, 4) == GL_ERR_INVALID           # no challenge
    assert _partial_products_rc(ctx, 8, 3, 5, 4) == GL_ERR_INVALID           # more than 4 challenges
    assert _partial_products_rc(ctx, 8, 3, 4, 4) == 0


# ------------------------------------------------------------------------------------------------ gl_quotient_add_permutation
def _commits(g, ctx, rng, log_n, r, n_ch, n_routed, degree, extra_wires=5):
    """random wires (more columns than n_routed), constants + sigmas (sigmas from column 3) and Z / partial-products commits"""
    n, n_chunks = 1 << log_n, -(-n_routed // degree)
    wires_b = g.PolynomialBatch.from_values(list(_field(rng, (max(n_routed + extra_wires, 4), n))), r, False, 0, ctx=ctx)
    sig_b = g.PolynomialBatch.from_values(list(_field(rng, (3 + n_routed + 2, n))), r, False, 0, ctx=ctx)
    zs_b = g.PolynomialBatch.from_values(list(_field(rng, (n_ch * n_chunks, n))), r, False, 0, ctx=ctx)
    return wires_b, sig_b, zs_b


# (log_n, rate_bits, n_ch, n_routed, degree): every n_ch 1..4 and every rate_bits 0..6; the last one is the wrapper circuit's
PERM_CASES = [(6, 0, 2, 16, 4), (4, 1, 1, 20, 2), (6, 2, 3, 40, 4), (10, 3, 4, 80, 8), (8, 4, 2, 80, 16), (5, 5, 1, 13, 4), (4, 6, 4, 80, 8),
              (16, 3, 2, 80, 8)]


@pytest.mark.gpu
@pytest.mark.parametrize("log_n,r,n_ch,n_routed,degree", PERM_CASES)
def test_permutation_terms_sweep(ctx, oc, log_n, r, n_ch, n_routed, degree):
    """the alpha-reduced permutation terms the kernel adds to a non-zero accumulator, against glo_vanishing_permutation at every leaf row
    (up to 2^16 rows); at 2^19 rows, the first and last point of each of the 2^r cosets of H (the last ones are the rows whose "next"
    point wraps) and 4096 random rows"""
    import plonky25_b200 as g
    rng = np.random.default_rng(8000 + 100 * log_n + 10 * r + n_ch)
    bits, R = log_n + r, 1 << (log_n + r)
    wires_b, sig_b, zs_b = _commits(g, ctx, rng, log_n, r, n_ch, n_routed, degree)
    k_is, betas, gammas, alphas = _field(rng, n_routed), _field(rng, n_ch, 0.5), _field(rng, n_ch, 0.5), _field(rng, n_ch, 0.5)
    quot = g.Quotient(wires_b, n_ch, ctx=ctx)
    quot.add_gate(*BASE_SUM, alphas)                                           # something underneath, so the kernel must add, not store
    before = quot.values()
    assert np.count_nonzero(before) > before.size // 2
    quot.add_permutation(sig_b, 3, zs_b, n_routed, degree, k_is, betas, gammas, alphas)
    got = _mod_sub(quot.values(), before).T                                    # [R][n_ch]
    quot.free()
    if R <= 1 << 16:
        rows = np.arange(R, dtype=np.uint64)
    else:
        edge = np.concatenate([np.arange(1 << r), np.arange(R - (1 << r), R)]).astype(np.uint64)
        rows = np.unique(np.concatenate([_bitrev(edge, bits), rng.integers(0, R, size=4096, dtype=np.uint64)]))
    want = po.vanishing_permutation(wires_b.merkle_tree.leaves, sig_b.merkle_tree.leaves, 3, zs_b.merkle_tree.leaves, rows, log_n, r,
                                    n_routed, degree, k_is, betas, gammas, alphas)
    got = got[rows.astype(np.int64)]
    bad = np.argwhere(got != want)
    assert bad.size == 0, f"{len(bad)} words differ, first (leaf row, challenge) {[(int(rows[i]), int(k)) for i, k in bad[:4]]}"
    for b in (wires_b, sig_b, zs_b):
        b.merkle_tree.free()


@pytest.mark.gpu
def test_add_permutation_refusals_leave_the_accumulator(ctx):
    """a Z batch with the wrong column count and a wires batch at rate_bits 7 are refused, and the accumulator is left as it was"""
    import plonky25_b200 as g
    rng = np.random.default_rng(8500)
    n_routed, degree, n_ch = 12, 4, 2
    k_is, betas, gammas, alphas = (_field(rng, m) for m in (n_routed, n_ch, n_ch, n_ch))
    ptr = lambda a: a.ctypes.data
    for log_n, r, extra_z in ((4, 3, 1), (2, 7, 0)):
        wires_b, sig_b, _ = _commits(g, ctx, rng, log_n, r, n_ch, n_routed, degree)
        zs_b = g.PolynomialBatch.from_values(list(_field(rng, (n_ch * 3 + extra_z, 1 << log_n))), r, False, 0, ctx=ctx)
        quot = g.Quotient(wires_b, n_ch, ctx=ctx)
        quot.add_gate(*BASE_SUM, alphas)
        before = quot.values()
        rc = ctx.lib.gl_quotient_add_permutation(ctx.handle, quot._h, sig_b.merkle_tree._h, 3, zs_b.merkle_tree._h, n_routed, degree,
                                                 ptr(k_is), ptr(betas), ptr(gammas), ptr(alphas))
        assert rc == (GL_ERR_INVALID if extra_z else GL_ERR_UNSUPPORTED), (log_n, r)
        assert np.array_equal(quot.values(), before)
        quot.free()
        for b in (wires_b, sig_b, zs_b):
            b.merkle_tree.free()


# ------------------------------------------------------------------------------------------------ gl_quotient_commit
# every n_ch 1..4 against every rate_bits 0..6 at small log_n with log_n + r >= 3 (N = 1 at (0, 3, 1), (0, 3, 4), (0, 4, 1), ...),
# then 2^12 at rate 4 with 4 challenges and the wrapper circuit's 2^16 at rate 3 with 2
QC_CASES = [(max(3 - r, 0) + (n_ch - 1) % 3, r, n_ch) for r in range(7) for n_ch in range(1, 5)] + [(12, 4, 4), (16, 3, 2)]


@pytest.mark.gpu
@pytest.mark.parametrize("log_n,r,n_ch", QC_CASES)
def test_quotient_commit_sweep(ctx, oc, log_n, r, n_ch):
    """acc / Z_H on the coset -> coset iFFT -> 2^r chunks per challenge -> from_coeffs commit, against glo_quotient_chunks and glo_commit.
    The accumulator holds permutation terms of random commits (they do not vanish on H); the tail is linear, so any values do."""
    import plonky25_b200 as g
    rng = np.random.default_rng(9000 + 100 * log_n + 10 * r + n_ch)
    n_routed, degree = (80, 8) if log_n >= 12 else (10, 4)
    h = min(2, log_n + r)
    wires_b, sig_b, zs_b = _commits(g, ctx, rng, log_n, r, n_ch, n_routed, degree)
    quot = g.Quotient(wires_b, n_ch, ctx=ctx)
    quot.add_permutation(sig_b, 3, zs_b, n_routed, degree, *(_field(rng, m, 0.5) for m in (n_routed, n_ch, n_ch, n_ch)))
    acc = quot.values()
    assert np.count_nonzero(acc) > acc.size // 2
    batch = quot.commit(h)
    quot.free()
    want = po.quotient_chunks(acc, log_n, r)
    got = batch.polynomials
    assert got.shape == want.shape == (n_ch << r, 1 << log_n)
    bad = np.argwhere(got != want)
    assert bad.size == 0, f"{len(bad)} coefficients differ, first (chunk row, coefficient) {bad[:4].tolist()}"
    assert np.array_equal(batch.merkle_tree.cap.hashes, oc.commit(want, r, h, is_coeffs=True, want=())["cap"])
    for b in (wires_b, sig_b, zs_b, batch):
        b.merkle_tree.free()


@pytest.mark.gpu
@pytest.mark.parametrize("log_n,r", [(0, 2), (1, 1), (2, 0)])
def test_quotient_commit_refuses_a_domain_below_8_points(ctx, log_n, r):
    import plonky25_b200 as g
    rng = np.random.default_rng(9500 + 10 * log_n + r)
    wires_b = g.PolynomialBatch.from_values(list(_field(rng, (4, 1 << log_n))), r, False, 0, ctx=ctx)
    quot = g.Quotient(wires_b, 1, ctx=ctx)
    quot.add_gate(*BASE_SUM, [3])
    cap, h = np.zeros(4, dtype=np.uint64), ctypes.c_uint64()
    assert ctx.lib.gl_quotient_commit(ctx.handle, quot._h, 0, cap.ctypes.data, ctypes.byref(h)) == GL_ERR_UNSUPPORTED
    quot.free()
    wires_b.merkle_tree.free()


# ------------------------------------------------------------------------------------------------ the whole argument at prover size
# (log_n, rate_bits, n_ch, n_routed, degree, tamper): degree <= 2^rate_bits, so the quotient has degree below 2^r N
IDENTITY_CASES = [(16, 3, 2, 80, 8, False), (12, 4, 4, 80, 16, False), (10, 1, 3, 20, 2, False), (10, 1, 3, 20, 2, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("log_n,r,n_ch,n_routed,degree,tamper", IDENTITY_CASES)
def test_verifier_identity_at_zeta(ctx, log_n, r, n_ch, n_routed, degree, tamper):
    """wires on a copy permutation -> gl_partial_products -> wires / constants+sigmas / Z commits -> gl_quotient_add_permutation ->
    gl_quotient_commit; then the verifier's check at a random zeta: Z_H(zeta) sum_c zeta^(cN) t_c(zeta) = sum_t alpha_k^t term_t(zeta)
    for every challenge, with every polynomial evaluated from its committed coefficients.  With one wire of one cycle changed the
    running product does not close, the terms do not vanish on H, and the identity fails."""
    import plonky25_b200 as g
    rng = np.random.default_rng(9900 + 100 * log_n + n_ch)
    n = 1 << log_n
    k_is = np.array([pow(7, j, P) for j in range(n_routed)], dtype=np.uint64)
    wires, sigmas = _copy_permutation(rng, n_routed, log_n, k_is, cycle_len=3)
    if tamper:
        j, i = int(rng.integers(n_routed)), int(rng.integers(n))
        wires[j, i] = (int(wires[j, i]) + 1) % P
    betas, gammas, alphas = _field(rng, n_ch, 0.5), _field(rng, n_ch, 0.5), _field(rng, n_ch, 0.5)
    k_nc = _noncanonical_form(rng, k_is)
    zs = g.partial_products_and_zs(list(wires), list(sigmas), k_nc, betas, gammas, degree, ctx=ctx)
    extra = _field(rng, (5, n))
    wires_b = g.PolynomialBatch.from_values(list(wires) + list(extra), r, False, 2, ctx=ctx)
    sig_b = g.PolynomialBatch.from_values(list(_field(rng, (3, n))) + list(sigmas), r, False, 2, ctx=ctx)
    zs_b = g.PolynomialBatch.from_values(list(zs), r, False, 2, ctx=ctx)
    quot = g.Quotient(wires_b, n_ch, ctx=ctx)
    quot.add_permutation(sig_b, 3, zs_b, n_routed, degree, k_nc, betas, gammas, alphas)
    t_b = quot.commit(2)
    quot.free()
    zeta = int(rng.integers(2, P, dtype=np.uint64))
    g_zeta = zeta * pow(GENERATOR, 1 << (32 - log_n), P) % P
    ev = lambda polys, x: [int(v) for v in oso.eval_ext(polys, (x, 0))[:, 0]]
    ew = ev(wires_b.polynomials[:n_routed], zeta)
    es = ev(sig_b.polynomials[3:3 + n_routed], zeta)
    ez, ezn = ev(zs_b.polynomials, zeta), ev(zs_b.polynomials, g_zeta)
    et = ev(t_b.polynomials, zeta)
    terms = go.vanishing_permutation_terms(ew, es, ez, ezn, zeta, _ints(k_is), _ints(betas), _ints(gammas), degree, log_n)
    z_h, zeta_n = (pow(zeta, n, P) - 1) % P, pow(zeta, n, P)
    holds = []
    for c in range(n_ch):
        t_zeta = 0
        for ch in reversed(range(1 << r)):
            t_zeta = (t_zeta * zeta_n + et[(c << r) + ch]) % P
        holds.append(z_h * t_zeta % P == go.reduce_with_powers(terms, _ints(alphas)[c]))
    if tamper:
        assert not any(holds), "the identity holds although the wires break the copy constraint"
    else:
        assert all(holds), f"Z_H(zeta) t(zeta) != vanishing(zeta) for challenges {[c for c in range(n_ch) if not holds[c]]}"
    for b in (wires_b, sig_b, zs_b, t_b):
        b.merkle_tree.free()
