"""plonky2.5_b200 — B200-native (sm_100a) commitment engine for the plonky2 prover that plonky2.5 drives.

Scope: exactly the hot path of SURVEY.md §8 — PolynomialBatch::from_values / from_coeffs (iNTT, coset LDE,
bit-reversed row-major leaves), Poseidon MerkleTree::new, FRI commit-phase folding — behind the C ABI of
include/gl_commit.h.  The directory name contains a dot, so import it as ``plonky25_b200`` (the shim module at the
repository root) or via importlib.
"""
from . import _lib  # noqa: F401
from . import sharded  # noqa: F401
from .api import (Challenger, Context, FriBatchInfo, FriOpeningBatch, FriOpenings, FriParams, FriProofHead, GlError, MerkleCap,  # noqa: F401
                  MerkleTree, OpeningSet, PolynomialBatch, commit_multi, eval_commitment, default_context, fri_committed_trees, fri_proof_of_work, fri_prover_query_rounds, prove_openings, reduction_arity_bits)
from .api import (GATE_COMPARISON, GATE_POSEIDON2, GATE_U32_ADD_MANY, GATE_U32_ARITHMETIC, GATE_U32_INTERLEAVE, GATE_U32_RANGE_CHECK,  # noqa: F401
                  GATE_U32_SUBTRACTION, GATE_UNINTERLEAVE_TO_B32, GATE_UNINTERLEAVE_TO_U32, Quotient, evaluate_gate_constraints, gate_shape,
                  partial_products_and_zs, poseidon2_gate_witness)
from .api import GATE_ARITHMETIC, GATE_BASE_SUM, GATE_CONSTANT, GATE_NOOP, GATE_PUBLIC_INPUT, SelectorsInfo  # noqa: F401
from .api import GATE_EXPONENTIATION, GATE_POSEIDON, GATE_RANDOM_ACCESS, poseidon_gate_witness, random_access_params  # noqa: F401
from .build import build  # noqa: F401

__all__ = ["Challenger", "Context", "FriBatchInfo", "FriOpeningBatch", "FriOpenings", "FriParams", "FriProofHead", "GlError", "MerkleCap",
           "MerkleTree", "OpeningSet", "PolynomialBatch", "commit_multi", "eval_commitment", "default_context", "fri_committed_trees", "fri_proof_of_work", "fri_prover_query_rounds", "prove_openings", "reduction_arity_bits", "build"]
