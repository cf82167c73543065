"""The wrapper-shaped prove pipeline of tests/wrapper_pipeline.py with the step prove() takes between zeta and alpha: compute the
OpeningSet (every committed polynomial at zeta, the Z polynomials also at g*zeta), then observe its FRI openings before alpha.

    run_product(g, ctx, cols, log_n, ...)   the product: OpeningSet.new on the device (gl_batch_eval), Challenger.observe_openings
    run_oracle(oc, cols, log_n, ...)        the CPU oracle: the host Horner of tests/opening_set_oracle.py on the oracle's coefficients

Both call wrapper_pipeline's own runners, so shapes, call order and every other proof byte come from the one pipeline; the step is
inserted where it belongs (product: at the top of prove_openings, before it draws alpha; oracle: right after the challenger hands out
zeta).  proof["openings"] holds the two FRI opening batches ([n][2] words each); `digest` hashes them after wrapper_pipeline.digest.
"""
import hashlib

import numpy as np

import opening_set_oracle
import wrapper_pipeline as wp

P = wp.P
NUM_CONSTANTS = 6     # commit #0 = 6 constants + 80 routed sigmas
NUM_CHALLENGES = 2    # commit #2 = the Z polynomial of each challenge, then the partial products


def generator(log_n):
    """the generator of the size-2^log_n subgroup"""
    return pow(1753635133440165772, 1 << (32 - log_n), P)


def oracle_openings(coeffs, zeta, log_n):
    """to_fri_openings() of OpeningSet::new on the host: [zeta batch (every polynomial of every commit), g*zeta batch (the Zs)]"""
    n_zs = min(NUM_CHALLENGES, len(coeffs[2]))
    zeta_batch = np.concatenate([opening_set_oracle.eval_ext(c, zeta) for c in coeffs])
    return [zeta_batch, opening_set_oracle.eval_ext(coeffs[2][:n_zs], wp._g_times(zeta, log_n))]


def digest(proof) -> str:
    h = hashlib.sha256(wp.digest(proof).encode())
    for batch in proof["openings"]:
        h.update(np.ascontiguousarray(batch, dtype=np.uint64).tobytes())
    return h.hexdigest()


class _ProductWithOpenings:
    """the package `g` as wrapper_pipeline.run_product sees it, with prove_openings preceded by OpeningSet::new + observe_openings"""

    def __init__(self, g, sink):
        self._g, self._sink = g, sink

    def __getattr__(self, name):
        return getattr(self._g, name)

    def prove_openings(self, instance, oracles, challenger, fri_params, **kw):
        zeta = instance[0].point
        cs, wires, zs, quotient = oracles
        oset = self._g.OpeningSet.new(zeta, generator(cs.degree_log), cs, wires, zs, quotient,
                                      min(NUM_CONSTANTS, cs.merkle_tree.leaf_len), min(NUM_CHALLENGES, zs.merkle_tree.leaf_len))
        fo = oset.to_fri_openings()
        challenger.observe_openings(fo)
        self._sink.extend(b.values.copy() for b in fo.batches)
        return self._g.prove_openings(instance, oracles, challenger, fri_params, **kw)


def run_product(g, ctx, cols, log_n, **kw):
    sink = []
    proof = wp.run_product(_ProductWithOpenings(g, sink), ctx, cols, log_n, **kw)
    proof["openings"] = sink
    return proof


class _ChallengerAfterZeta:
    """the oracle's challenger; right after the first extension challenge (zeta) it calls `hook(challenger, zeta)`"""

    def __init__(self, inner, hook):
        self._inner, self._hook = inner, hook

    def __getattr__(self, name):
        return getattr(self._inner, name)

    def get_extension_challenge(self):
        e = self._inner.get_extension_challenge()
        if self._hook is not None:
            hook, self._hook = self._hook, None
            hook(self._inner, e)
        return e


class _OracleWithOpenings:
    """the oracle as wrapper_pipeline.run_oracle sees it: remembers each commit's coefficients, and observes the openings after zeta"""

    def __init__(self, oc, log_n, sink):
        self._oc, self._log_n, self._sink, self._coeffs = oc, log_n, sink, []

    def __getattr__(self, name):
        return getattr(self._oc, name)

    def commit(self, *a, **kw):
        cm = self._oc.commit(*a, **kw)
        self._coeffs.append(cm["coeffs"])
        return cm

    def new_challenger(self):
        return _ChallengerAfterZeta(self._oc.new_challenger(), self._observe_openings)

    def _observe_openings(self, ch, zeta):
        openings = oracle_openings(self._coeffs, zeta, self._log_n)
        for batch in openings:
            ch.observe_extension_elements(batch)
        self._sink.extend(openings)


def run_oracle(oc, cols, log_n, **kw):
    sink = []
    proof = wp.run_oracle(_OracleWithOpenings(oc, log_n, sink), cols, log_n, **kw)
    proof["openings"] = sink
    return proof
