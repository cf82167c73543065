"""OpeningSet::new on the device (gl_batch_eval): every committed polynomial at zeta, the Z commit also at g*zeta, and the transcript step
that observes the openings before alpha.  CPU: the C oracle's evaluation, the wrapper pipeline's proof with openings under the verifier
restatement, and the C++ mirror's host logic on the ABI double.  GPU: parity with the oracle, identities that need no oracle, the error
paths, the whole wrapper-shaped proof and the C++ mirror on the real library."""
import os
import subprocess

import numpy as np
import pytest

import opening_set_oracle as oso
import opening_set_pipeline as osp
import wrapper_pipeline as wp
from oracle_c import P, splitmix_columns

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CPP_SRC = os.path.join(ROOT, "tests", "cpp", "opening_set_test.cpp")
W = 1753635133440165772   # 2^32nd root of unity


def _cxx(args):
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    env = dict(os.environ)
    env.pop("CC", None); env.pop("CXX", None)
    subprocess.run([cxx, "-std=c++17", "-O2", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), *args, "-pthread"],
                   check=True, env=env)


def _rand_point(rng, canonical=True):
    hi = P if canonical else 1 << 64
    return (int(rng.integers(0, hi, dtype=np.uint64)), int(rng.integers(0, hi, dtype=np.uint64)))


# ------------------------------------------------------------------------------------------------------------------------------- CPU
def test_oracle_eval_ext_matches_python_oracle():
    import gl_oracle as o
    rng = np.random.default_rng(5)
    for n_polys, n in ((1, 1), (3, 8), (5, 33)):
        polys = splitmix_columns(11 + n, n_polys, n, canonical=False)      # raw words, some >= p
        for canonical in (True, False):
            z = _rand_point(rng, canonical)
            got = oso.eval_ext(polys, z)
            for j in range(n_polys):
                want = o.ext_eval_poly_ext([(int(c) % P, 0) for c in polys[j]], (z[0] % P, z[1] % P))
                assert tuple(int(v) for v in got[j]) == want
    assert oso.eval_ext(np.zeros((0, 4), dtype=np.uint64), (1, 2)).shape == (0, 2)


def _verify(oc, proof, log_n, r, h, arities, pow_bits, openings):
    import gl_oracle as o
    import fri_verifier as fv
    commits = [oc.commit(c, r, h, is_coeffs=wp.IS_COEFFS[k], want=()) for k, c in enumerate(wp.make_columns(log_n))]
    ch = o.Challenger()
    ch.observe_elements([int(v) for v in wp.PREFIX])
    for cm in commits:
        ch.observe_cap(cm["cap"].tolist())
    zeta = ch.get_extension_challenge()
    for batch in openings:                                   # observe_openings(&openings.to_fri_openings())
        for e in batch:
            ch.observe_extension_element((int(e[0]), int(e[1])))
    all_polys, zs = wp.instance_for(wp.WIDTHS)
    batches = [(zeta, all_polys), (wp._g_times(zeta, log_n), zs)]
    opened = [[(int(e[0]), int(e[1])) for e in batch] for batch in openings]
    rounds = [{"x_index": x,
               "initial_trees_proof": [([int(v) for v in row], [[int(w) for w in s] for s in sib]) for row, sib in rnd["initial"]],
               "steps": [{"evals": [(int(e[0]), int(e[1])) for e in ev], "merkle_proof": [[int(w) for w in s] for s in sib]}
                         for ev, sib in rnd["steps"]]}
              for x, rnd in zip(proof["query_indices"], proof["query_rounds"])]
    fv.verify_fri_proof(batches=batches, opened_values=opened, initial_caps=[cm["cap"].tolist() for cm in commits],
                        commit_caps=[c.tolist() for c in proof["commit_phase_caps"]],
                        final_poly=[(int(c[0]), int(c[1])) for c in proof["final_poly"]], pow_witness=proof["pow_witness"],
                        query_rounds=rounds, challenger=ch, reduction_arity_bits=list(arities), log_n=log_n, rate_bits=r, pow_bits=pow_bits)


def test_oracle_proof_with_openings_passes_the_verifier(oc):
    log_n, r, h, arities, pow_bits = 6, 3, 4, (4,), 4
    cols = wp.make_columns(log_n)
    proof = osp.run_oracle(oc, cols, log_n, r=r, h=h, arities=arities, pow_bits=pow_bits, n_queries=5)
    openings = proof["openings"]
    assert [b.shape for b in openings] == [(sum(wp.WIDTHS), 2), (osp.NUM_CHALLENGES, 2)]
    _verify(oc, proof, log_n, r, h, arities, pow_bits, openings)
    # the openings are bound to the proof: the verifier sees a different alpha, the reduced openings no longer match
    bad = [b.copy() for b in openings]
    bad[0][100, 1] = (int(bad[0][100, 1]) + 1) % P
    with pytest.raises(AssertionError):
        _verify(oc, proof, log_n, r, h, arities, pow_bits, bad)
    # observing the openings moves alpha and everything after it
    plain = wp.run_oracle(oc, cols, log_n, r=r, h=h, arities=arities, pow_bits=pow_bits, n_queries=5)
    assert "openings" not in plain and wp.digest(plain) != wp.digest(proof)


def test_cpp_opening_set_mirror_on_abi_double(tmp_path):
    from oracle_c import build_oracle
    ora = build_oracle()
    exe = str(tmp_path / "opening_set_test_double")
    horner = oso.build()
    _cxx([CPP_SRC, os.path.join(ROOT, "tests", "cpp", "abi_test_double.cpp"), os.path.join(ROOT, "tests", "cpp", "abi_test_double_batch_eval.cpp"),
          "-o", exe, "-L", os.path.dirname(ora), "-lgl_oracle", "-Wl,-rpath," + os.path.dirname(ora),
          "-L", os.path.dirname(horner), "-leval_ext_oracle", "-Wl,-rpath," + os.path.dirname(horner)])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "ALL OK" in r.stdout, r.stdout[-3000:] + r.stderr[-2000:]


# ------------------------------------------------------------------------------------------------------------------------------- GPU
def _commit(g, ctx, cols, is_coeffs=False, r=1, h=0):
    fn = g.PolynomialBatch.from_coeffs if is_coeffs else g.PolynomialBatch.from_values
    return fn(list(cols), r, False, h, ctx=ctx)


@pytest.mark.gpu
@pytest.mark.parametrize("width", [1, 7, 135, 86, 20, 16])
@pytest.mark.parametrize("log_n", [0, 1, 3, 7, 10, 16])
def test_batch_eval_matches_oracle(ctx, width, log_n):
    import plonky25_b200 as g
    rng = np.random.default_rng(1000 * log_n + width)
    cols = splitmix_columns(log_n * 31 + width, width, 1 << log_n, canonical=False)
    for is_coeffs in (False, True):
        b = _commit(g, ctx, cols, is_coeffs)
        coeffs = cols if is_coeffs else b.polynomials
        z1, z2 = _rand_point(rng, canonical=False), _rand_point(rng)
        one = g.eval_commitment(b, [z1])
        assert one.shape == (1, width, 2)
        assert np.array_equal(one[0], oso.eval_ext(coeffs, z1))
        two = g.eval_commitment(b, [z2, z1])
        assert np.array_equal(two[0], oso.eval_ext(coeffs, z2)) and np.array_equal(two[1], one[0])
        b.merkle_tree.free()


@pytest.mark.gpu
def test_batch_eval_large_batch(ctx):
    """one 2^20 x 135 commit at two points (several sub-chunks per CTA)"""
    import plonky25_b200 as g
    cols = splitmix_columns(77, 135, 1 << 20)
    b = _commit(g, ctx, cols, r=1, h=4)
    z = [(12345678901234567, 98765432109876543), (P - 3, 5)]
    got = g.eval_commitment(b, z)
    coeffs = b.polynomials
    for p in range(2):
        assert np.array_equal(got[p], oso.eval_ext(coeffs, z[p]))
    b.merkle_tree.free()


@pytest.mark.gpu
def test_batch_eval_quotient_commit(ctx):
    import plonky25_b200 as g
    log_n, n_ch = 6, 2
    wires = _commit(g, ctx, splitmix_columns(3, 135, 1 << log_n), r=3)
    q = g.Quotient(wires, n_ch)
    q.add_gate(g.GATE_POSEIDON2, 0, splitmix_columns(4, 1, n_ch).reshape(-1))
    qb = q.commit(0)
    coeffs = qb.polynomials
    z = (987654321, 123456789)
    assert np.array_equal(g.eval_commitment(qb, [z])[0], oso.eval_ext(coeffs, z))
    q.free(); qb.merkle_tree.free(); wires.merkle_tree.free()


@pytest.mark.gpu
@pytest.mark.parametrize("width,log_n", [(135, 10), (20, 4), (1, 0)])
def test_batch_eval_identities(ctx, width, log_n):
    """no oracle: values on the subgroup are the committed values, on the LDE coset they are the leaves, at 0 they are coefficient row 0"""
    import plonky25_b200 as g
    n, r = 1 << log_n, 2
    cols = splitmix_columns(5 + width, width, n)
    b = _commit(g, ctx, cols, r=r)
    wn = pow(W, 1 << (32 - log_n), P)
    for i in sorted({0, 1, n // 2, n - 1} & set(range(n))):
        assert np.array_equal(g.eval_commitment(b, [(pow(wn, i, P), 0)])[0][:, 0], cols[:, i])
        assert not g.eval_commitment(b, [(pow(wn, i, P), 0)])[0][:, 1].any()
    wr = pow(W, 1 << (32 - log_n - r), P)
    R = n << r
    for i in sorted({0, 3, R - 1} & set(range(R))):
        x = 7 * pow(wr, int(format(i, f"0{log_n + r}b")[::-1], 2), P) % P
        assert np.array_equal(g.eval_commitment(b, [(x, 0)])[0][:, 0], b.merkle_tree.get(i))
    assert np.array_equal(g.eval_commitment(b, [(0, 0)])[0][:, 0], b.polynomials[:, 0])
    b.merkle_tree.free()


@pytest.mark.gpu
def test_batch_eval_error_paths(ctx):
    import ctypes
    import plonky25_b200 as g
    from plonky25_b200 import _lib
    lib = ctx.lib
    b = _commit(g, ctx, splitmix_columns(9, 4, 16))
    h = b.merkle_tree._h
    pts = np.array([1, 2, 3, 4, 5, 6], dtype=np.uint64)
    out = np.zeros(3 * 4 * 2, dtype=np.uint64)
    p, o = pts.ctypes.data_as(ctypes.c_void_p), out.ctypes.data_as(ctypes.c_void_p)
    assert lib.gl_batch_eval(ctx.handle, h, p, 1, o) == _lib.GL_OK
    assert lib.gl_batch_eval(ctx.handle, 987654321, p, 1, o) == _lib.GL_ERR_HANDLE
    assert lib.gl_batch_eval(ctx.handle, h, None, 1, o) == _lib.GL_ERR_INVALID
    assert lib.gl_batch_eval(ctx.handle, h, p, 1, None) == _lib.GL_ERR_INVALID
    assert lib.gl_batch_eval(ctx.handle, h, p, 0, o) == _lib.GL_ERR_INVALID
    assert lib.gl_batch_eval(ctx.handle, h, p, 3, o) == _lib.GL_ERR_UNSUPPORTED
    with pytest.raises(ValueError, match="tree has no coefficients"):
        g.eval_commitment(g.PolynomialBatch(ctx, g.MerkleTree.new(splitmix_columns(1, 16, 3), 0, ctx=ctx), 3), [(1, 2)])
    b.merkle_tree.free()
    ctx2 = g.Context(0)
    try:
        _, shards = g.commit_multi([ctx, ctx2], list(splitmix_columns(2, 8, 16)), 1, 1)
        for c, t in zip((ctx, ctx2), shards):
            assert c.lib.gl_batch_eval(c.handle, t._h, p, 1, o) == _lib.GL_ERR_INVALID
            assert "tree has no coefficients" in c.lib.gl_ctx_last_error(c.handle).decode()
            t.free()
    finally:
        ctx2.close()


@pytest.mark.gpu
@pytest.mark.parametrize("log_n,arities,pow_bits", [(10, (4, 4), 8), (16, wp.ARITIES, wp.POW_BITS)])
def test_wrapper_pipeline_with_openings_matches_oracle(ctx, oc, log_n, arities, pow_bits):
    import plonky25_b200 as g
    cols = wp.make_columns(log_n)
    want = osp.run_oracle(oc, cols, log_n, arities=arities, pow_bits=pow_bits)
    got = osp.run_product(g, ctx, cols, log_n, arities=arities, pow_bits=pow_bits)
    assert len(got["openings"]) == 2
    for a, b in zip(got["openings"], want["openings"]):
        assert np.array_equal(a, b)
    for key in ("commit_caps", "commit_phase_caps"):
        for a, b in zip(got[key], want[key]):
            assert np.array_equal(a, b)
    assert np.array_equal(got["final_poly"], want["final_poly"])
    assert got["pow_witness"] == want["pow_witness"] and got["query_indices"] == want["query_indices"]
    for ra, rb in zip(got["query_rounds"], want["query_rounds"]):
        for (r1, s1), (r2, s2) in zip(ra["initial"], rb["initial"]):
            assert np.array_equal(r1, r2) and np.array_equal(s1, s2)
        for (e1, s1), (e2, s2) in zip(ra["steps"], rb["steps"]):
            assert np.array_equal(e1, e2) and np.array_equal(s1, s2)
    assert osp.digest(got) == osp.digest(want)
    if log_n == 10:
        _verify(oc, got, log_n, 3, 4, arities, pow_bits, got["openings"])


@pytest.mark.gpu
def test_cpp_opening_set_mirror_on_gpu(tmp_path):
    import plonky25_b200 as g
    lib = g.build()
    exe = str(tmp_path / "opening_set_test")
    _cxx([CPP_SRC, "-o", exe, "-L", os.path.dirname(lib), "-lgl_commit", "-Wl,-rpath," + os.path.dirname(lib)])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "ALL OK" in r.stdout, r.stdout[-3000:] + r.stderr[-2000:]
