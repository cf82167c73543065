"""ctypes binding of libgl_commit.so — exactly the C ABI in include/gl_commit.h, nothing else.

There is no fallback: if the CUDA library is missing or no device is present, loading / context creation raises.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_size_t, c_uint32, c_uint64, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libgl_commit.so")

GL_OK, GL_ERR_INVALID, GL_ERR_CUDA, GL_ERR_OOM, GL_ERR_HANDLE, GL_ERR_UNSUPPORTED = 0, -1, -2, -3, -4, -5
GL_PART_COEFFS, GL_PART_LEAVES, GL_PART_DIGESTS, GL_PART_CAP = 0, 1, 2, 3
GL_GATE_POSEIDON2, GL_GATE_U32_ARITHMETIC = 0, 1
STAGES = ("h2d", "transpose", "intt", "lde", "leaf_hash", "tree", "d2h")


class TreeInfo(ctypes.Structure):
    _fields_ = [("n_leaves", c_uint64), ("leaf_len", c_uint32), ("cap_height", c_uint32), ("degree_log", c_uint32),
                ("rate_bits", c_uint32), ("has_coeffs", c_uint32), ("pitch", c_uint32)]


class StreamPlan(ctypes.Structure):
    """gl_stream_plan_t (include/gl_commit.h): the streamed coset-sharded commit of one rank"""
    _fields_ = [("n_cols", c_uint32), ("log_n", c_uint32), ("rate_bits", c_uint32), ("cap_height", c_uint32), ("n_peers", c_uint32),
                ("self", c_uint32), ("group_width", c_uint32), ("leaf_pitch", c_uint32), ("epoch", c_uint64)]


u64p = POINTER(c_uint64)

# name -> (restype, argtypes); every symbol include/gl_commit.h declares
SIGNATURES = {
    "gl_abi_version": (c_int, []),
    "gl_strerror": (c_char_p, [c_int]),
    "gl_device_count": (c_int, []),
    "gl_ctx_create": (c_int, [POINTER(c_void_p), c_int]),
    "gl_ctx_destroy": (None, [c_void_p]),
    "gl_ctx_last_error": (c_char_p, [c_void_p]),
    "gl_ctx_stream": (c_uint64, [c_void_p]),
    "gl_commit": (c_int, [c_void_p, POINTER(c_void_p), c_uint32, c_uint32, c_uint32, c_uint32, c_int,
                          c_void_p, c_void_p, c_void_p, c_void_p, POINTER(c_uint64)]),
    "gl_commit_multi": (c_int, [POINTER(c_void_p), c_uint32, POINTER(c_void_p), c_uint32, c_uint32, c_uint32, c_uint32, c_int, c_void_p,
                                POINTER(c_uint64)]),
    "gl_merkle_new": (c_int, [c_void_p, c_void_p, c_uint64, c_uint32, c_uint32, c_void_p, c_void_p, POINTER(c_uint64)]),
    "gl_tree_info": (c_int, [c_void_p, c_uint64, POINTER(TreeInfo)]),
    "gl_tree_get": (c_int, [c_void_p, c_uint64, c_uint64, c_void_p]),
    "gl_tree_prove": (c_int, [c_void_p, c_uint64, c_uint64, c_void_p]),
    "gl_tree_open_batch": (c_int, [c_void_p, c_uint64, c_void_p, c_uint32, c_void_p, c_void_p]),
    "gl_tree_get_lde_values": (c_int, [c_void_p, c_uint64, c_uint64, c_uint64, c_void_p]),
    "gl_tree_read": (c_int, [c_void_p, c_uint64, c_int, c_void_p]),
    "gl_tree_free": (c_int, [c_void_p, c_uint64]),
    "gl_fri_begin": (c_int, [c_void_p, c_void_p, c_void_p, c_uint64, c_uint32, c_uint32, POINTER(c_uint64)]),
    "gl_fri_commit_layer": (c_int, [c_void_p, c_uint64, c_uint32, c_void_p, c_void_p, c_void_p, POINTER(c_uint64)]),
    "gl_fri_fold": (c_int, [c_void_p, c_uint64, c_void_p]),
    "gl_fri_final_poly": (c_int, [c_void_p, c_uint64, c_void_p, POINTER(c_uint64)]),
    "gl_fri_end": (c_int, [c_void_p, c_uint64]),
    "gl_openings_begin": (c_int, [c_void_p, c_uint32, POINTER(c_uint64)]),
    "gl_openings_add_batch": (c_int, [c_void_p, c_uint64, c_void_p, c_void_p, c_uint32, c_void_p, c_void_p, c_void_p]),
    "gl_openings_final_poly": (c_int, [c_void_p, c_uint64, c_void_p]),
    "gl_openings_lde": (c_int, [c_void_p, c_uint64, c_uint32, c_uint32, POINTER(c_uint64)]),
    "gl_openings_end": (c_int, [c_void_p, c_uint64]),
    "gl_batch_eval": (c_int, [c_void_p, c_uint64, c_void_p, c_uint32, c_void_p]),
    "gl_fri_read": (c_int, [c_void_p, c_uint64, c_void_p, c_void_p, POINTER(c_uint64)]),
    "gl_gate_num_wires": (c_int, [c_int, c_uint32]),
    "gl_gate_num_constraints": (c_int, [c_int, c_uint32]),
    "gl_gate_num_constants": (c_int, [c_int, c_uint32]),
    "gl_gate_eval_rows": (c_int, [c_void_p, c_int, c_uint32, c_void_p, c_uint64, c_void_p]),
    "gl_gate_eval_rows_with_constants": (c_int, [c_void_p, c_int, c_uint32, c_void_p, c_void_p, c_void_p, c_uint64, c_void_p]),
    "gl_quotient_begin": (c_int, [c_void_p, c_uint64, c_uint32, POINTER(c_uint64)]),
    "gl_quotient_add_gate": (c_int, [c_void_p, c_uint64, c_int, c_uint32, c_void_p, c_uint32, c_uint64, c_uint32]),
    "gl_quotient_add_gates": (c_int, [c_void_p, c_uint64, c_void_p, c_void_p, c_uint32, c_void_p, c_void_p, c_uint32, c_uint32, c_uint64, c_uint32,
                                      c_void_p, c_void_p, c_uint32]),
    "gl_quotient_add_permutation": (c_int, [c_void_p, c_uint64, c_uint64, c_uint32, c_uint64, c_uint32, c_uint32, c_void_p, c_void_p, c_void_p, c_void_p]),
    "gl_quotient_read": (c_int, [c_void_p, c_uint64, c_void_p]),
    "gl_quotient_commit": (c_int, [c_void_p, c_uint64, c_uint32, c_void_p, POINTER(c_uint64)]),
    "gl_quotient_end": (c_int, [c_void_p, c_uint64]),
    "gl_ctx_aux_ms": (c_int, [c_void_p, POINTER(c_float)]),
    "gl_poseidon2_gate_witness": (c_int, [c_void_p, c_void_p, c_uint64, c_void_p]),
    "gl_poseidon_gate_witness": (c_int, [c_void_p, c_void_p, c_uint64, c_void_p]),
    "gl_partial_products": (c_int, [c_void_p, POINTER(c_void_p), POINTER(c_void_p), c_uint32, c_uint32, c_void_p, c_void_p, c_void_p, c_uint32,
                                    c_uint32, c_void_p]),
    "gl_fri_pow": (c_int, [c_void_p, c_void_p, c_void_p, c_uint32, c_uint32, POINTER(c_uint64)]),
    "gl_poseidon_absorb": (c_int, [c_void_p, c_void_p, c_void_p, c_uint32]),
    "gl_poseidon_permute": (c_int, [c_void_p, c_void_p, c_uint64]),
    "gl_dev_commit": (c_int, [c_void_p, c_void_p, c_uint64, c_uint32, c_uint32, c_uint32, c_uint32, c_int, c_void_p,
                              POINTER(c_uint64)]),
    "gl_dev_lde": (c_int, [c_void_p, c_void_p, c_uint64, c_uint32, c_uint32, c_uint32, c_int, c_void_p, c_uint32, c_void_p]),
    "gl_dev_lde_scatter": (c_int, [c_void_p, c_void_p, c_uint64, c_uint32, c_uint32, c_uint32, c_int, POINTER(c_void_p), c_uint32,
                                   c_uint32, c_uint32, c_void_p, c_uint32, c_uint32]),
    "gl_lde_scatter": (c_int, [c_void_p, POINTER(c_void_p), c_uint32, c_uint32, c_uint32, c_int, POINTER(c_void_p), c_uint32,
                               c_uint32, c_uint32, c_void_p, c_uint32, c_uint32]),
    "gl_dev_intt": (c_int, [c_void_p, c_void_p, c_uint64, c_uint32, c_uint32, c_int, c_void_p, c_uint32]),
    "gl_intt_host": (c_int, [c_void_p, POINTER(c_void_p), c_uint32, c_uint32, c_int, c_void_p, c_uint32]),
    "gl_dev_lde_own_cosets": (c_int, [c_void_p, POINTER(c_void_p), POINTER(c_void_p), POINTER(c_uint32), POINTER(c_uint32), POINTER(c_uint32),
                                      c_uint32, c_uint32, c_uint32, c_uint32, c_void_p, c_uint32]),
    "gl_stream_plan_sizes": (c_int, [POINTER(StreamPlan), POINTER(c_uint64), POINTER(c_uint64), POINTER(c_uint32), POINTER(c_uint32)]),
    "gl_commit_coset_stream": (c_int, [c_void_p, POINTER(StreamPlan), POINTER(c_void_p), c_int, POINTER(c_void_p), c_void_p, c_void_p, c_void_p,
                                       c_void_p]),
    "gl_dev_ipc_alloc": (c_int, [c_void_p, c_uint64, POINTER(c_void_p), c_void_p]),
    "gl_dev_ipc_open": (c_int, [c_void_p, c_void_p, POINTER(c_void_p)]),
    "gl_dev_ipc_close": (c_int, [c_void_p, c_void_p]),
    "gl_dev_ipc_free": (c_int, [c_void_p, c_void_p]),
    "gl_dev_alloc": (c_int, [c_void_p, c_uint64, POINTER(c_void_p)]),
    "gl_dev_free": (c_int, [c_void_p, c_void_p]),
    "gl_dev_upload": (c_int, [c_void_p, c_void_p, c_void_p, c_uint64]),
    "gl_dev_download": (c_int, [c_void_p, c_void_p, c_void_p, c_uint64]),
    "gl_dev_repack": (c_int, [c_void_p, c_void_p, c_uint32, c_uint32, c_uint64, c_void_p, c_uint32, c_uint32]),
    "gl_dev_merkle": (c_int, [c_void_p, c_void_p, c_uint64, c_uint32, c_uint32, c_uint32, c_void_p, c_void_p]),
    "gl_ctx_stage_times": (c_int, [c_void_p, POINTER(c_float), POINTER(c_uint32)]),
    "gl_microbench": (c_int, [c_void_p, c_int, c_uint32, POINTER(c_double)]),
    "gl_field_op": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_uint64]),
    "gl_host_alloc": (c_void_p, [c_size_t]),
    "gl_host_free": (None, [c_void_p]),
}

_lib = None


def load() -> ctypes.CDLL:
    """dlopen the in-tree library and bind every symbol.  Raises if the library has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: build it with `python plonky2.5_b200/build.py` "
                           "(there is no CPU fallback for the commitment path)")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)   # AttributeError if the ABI and the header drift apart
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
