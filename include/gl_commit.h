/*
 * gl_commit.h — C ABI of libgl_commit: the B200-native (sm_100a) replacement for the commitment hot path of the
 * plonky2 prover that plonky2.5 drives (PolynomialBatch::from_values / from_coeffs, MerkleTree::new,
 * fri_committed_trees; and, next to it, the front half of prove_openings, the proof-of-work grind and the query-round
 * openings, so that the committed data never has to leave the device).  This is the drop-in boundary: plain C, `uint64_t` Goldilocks words (little-endian,
 * GoldilocksField is #[repr(transparent)] u64; inputs may be non-canonical, outputs are always canonical),
 * integer status returns, no unwinding across the boundary, no torch types.
 *
 * The reference reaches this path only through (file:line under /root/reference):
 *     src/p3/mod.rs:250   builder.build::<C>()  -> plonky2 circuit_builder.rs · build      -> from_values (commit #0)
 *     src/p3/mod.rs:260   data.prove(pw)        -> plonky2 plonk/prover.rs                 -> from_values x2, from_coeffs,
 *                                                  fri/oracle.rs · prove_openings -> fri/prover.rs · fri_committed_trees
 * (and the 23 other prove/verify pairs listed in SURVEY.md §4).  The upstream functions live in the un-vendored crate
 * plonky2 @ 3de92d9ed1721cec133e4e1e1b3ec7facb756ccf (Cargo.toml:15-19); each entry point below names the upstream
 * item it replaces.  The Rust binding a maintainer would add is shown in INTEGRATION.md.
 *
 * Threading: every call takes the context's mutex; calls on one context are serialised, distinct contexts are
 * independent (one context per prover thread is the intended use under `cargo test`'s parallel tests).
 * All calls are synchronous: on return the outputs are visible to the host.
 * There is NO CPU fallback: without a CUDA device gl_ctx_create fails with GL_ERR_CUDA.
 */
#ifndef GL_COMMIT_H
#define GL_COMMIT_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct gl_ctx gl_ctx;
typedef uint64_t gl_handle; /* device-resident object id (tree / batch / fri state); 0 is never valid */

enum {
    GL_OK = 0,
    GL_ERR_INVALID = -1,     /* argument violates an upstream assert (message via gl_ctx_last_error)            */
    GL_ERR_CUDA = -2,        /* CUDA runtime error / no device                                                   */
    GL_ERR_OOM = -3,         /* device or host allocation failed                                                 */
    GL_ERR_HANDLE = -4,      /* unknown handle                                                                   */
    GL_ERR_UNSUPPORTED = -5  /* shape outside what the kernels support (e.g. log_n + rate_bits > 32)             */
};

#define GL_ABI_VERSION 2
int gl_abi_version(void);
const char* gl_strerror(int code);

/* number of CUDA devices visible to the process (0 without a driver/device) */
int gl_device_count(void);

/* ---- context --------------------------------------------------------------------------------------------- */
int gl_ctx_create(gl_ctx** out, int device);
void gl_ctx_destroy(gl_ctx* ctx);
const char* gl_ctx_last_error(gl_ctx* ctx);
/* the CUDA stream all work of this context is enqueued on (cudaStream_t as integer) — for event timing */
uint64_t gl_ctx_stream(gl_ctx* ctx);

/* ---- PolynomialBatch::from_values / from_coeffs  (plonky2 fri/oracle.rs) ------------------------------------
 * cols          n_cols host pointers, each 2^log_n words: Vec<PolynomialValues<F>> (input_is_coeffs = 0) or
 *               Vec<PolynomialCoeffs<F>> (input_is_coeffs = 1) without a copy.  blinding is always false here.
 * out_coeffs    n_cols * N words, column-major, canonical (PolynomialBatch::polynomials); NULL = do not copy back
 * out_leaves    R * n_cols words row-major, row i = LDE point index bitrev(i) (MerkleTree::leaves); NULL = keep on device
 * out_digests   2*(R - 2^cap_height)*4 words, plonky2 interleaved layout (MerkleTree::digests); NULL = keep on device
 * out_cap       2^cap_height * 4 words (MerkleTree::cap), always written
 * out_batch     if non-NULL receives a handle to the device-resident batch (free with gl_tree_free); if NULL the
 *               device copy is released before returning.
 * Errors mirror upstream asserts: cap_height > log2(R) -> GL_ERR_INVALID ("cap_height should be at most
 * log2(leaves.len())"); n_cols == 0 -> GL_ERR_INVALID.
 */
int gl_commit(gl_ctx* ctx, const uint64_t* const* cols, uint32_t n_cols, uint32_t log_n, uint32_t rate_bits,
              uint32_t cap_height, int input_is_coeffs, uint64_t* out_coeffs, uint64_t* out_leaves,
              uint64_t* out_digests, uint64_t* out_cap, gl_handle* out_batch);

/* ---- the same commit on several GPUs from ONE process (CircuitData::prove is one process; BASELINE north star: columns sharded
 * across the GPUs of a box for the LDE, redistributed column->row over NVLink, hashed into per-GPU subtrees whose roots form the cap).
 * ctxs: n_ctx distinct contexts (a power of two <= 16, normally one per device; 2^cap_height >= n_ctx, n_cols >= n_ctx).  Context g
 * runs the iNTT + LDE of its column slice, receives leaf rows [g*R/n_ctx, (g+1)*R/n_ctx) from all contexts and hashes them.
 * out_cap: 2^cap_height * 4 words.  out_trees[g]: handle ON ctxs[g] of a device-resident tree over that leaf range with
 * cap_height - log2(n_ctx): leaf row i of the batch is gl_tree_get(ctxs[i / (R/n_ctx)], out_trees[i / (R/n_ctx)], i % (R/n_ctx)),
 * and gl_tree_prove on it returns exactly MerkleTree::prove(i) (the subtree roots are cap entries, so no path crosses contexts).
 * The shard trees carry no coefficient matrix (gl_tree_read(GL_PART_COEFFS) is refused) and gl_tree_get_lde_values does not
 * apply to them.  All contexts are locked for the duration of the call; status and message are reported through ctxs[0].
 * With TWO contexts on two devices (and 2 <= 2^rate_bits) the call runs the streamed coset plan (gl_commit_coset_stream below: column
 * groups dealt cyclically, per wave copy -> iNTT -> ticket -> peer pulls -> own cosets -> leaf sponge, no barrier between the first wave
 * and the cap); otherwise the column->row shipment described above (at 8 devices in ONE process the streamed plan is slower than the
 * shipment, see DESIGN.md §6).
 * Tested bit-exact against the oracle with several contexts on one device and with one device per context (tests/test_gpu_parity.py
 * spreads the contexts over every visible GPU; bench.py --gpus N --single-process times it).                                      */
int gl_commit_multi(gl_ctx* const* ctxs, uint32_t n_ctx, const uint64_t* const* cols, uint32_t n_cols, uint32_t log_n, uint32_t rate_bits,
                    uint32_t cap_height, int input_is_coeffs, uint64_t* out_cap, gl_handle* out_trees);

/* ---- MerkleTree::new  (plonky2 hash/merkle_tree.rs) ---------------------------------------------------------
 * leaves: n_leaves rows of leaf_len words, packed row-major on the host.  n_leaves must be a power of two. */
int gl_merkle_new(gl_ctx* ctx, const uint64_t* leaves, uint64_t n_leaves, uint32_t leaf_len, uint32_t cap_height,
                  uint64_t* out_digests, uint64_t* out_cap, gl_handle* out_tree);

/* ---- device-resident trees / batches: MerkleTree::get, MerkleTree::prove, PolynomialBatch::get_lde_values ---- */
typedef struct {
    uint64_t n_leaves;    /* R */
    uint32_t leaf_len;    /* n_cols */
    uint32_t cap_height;
    uint32_t degree_log;  /* log_n   (0 for bare trees) */
    uint32_t rate_bits;   /*         (0 for bare trees) */
    uint32_t has_coeffs;
    uint32_t pitch;       /* device row pitch in words */
} gl_tree_info_t;
int gl_tree_info(gl_ctx* ctx, gl_handle tree, gl_tree_info_t* out);
int gl_tree_get(gl_ctx* ctx, gl_handle tree, uint64_t leaf_index, uint64_t* out_row /* leaf_len */);
/* siblings bottom-up, (log2(n_leaves) - cap_height) * 4 words — MerkleProof::siblings */
int gl_tree_prove(gl_ctx* ctx, gl_handle tree, uint64_t leaf_index, uint64_t* out_siblings);
/* gl_tree_get + gl_tree_prove for n leaf indices in one launch and two copies (the FRI query rounds open 28 indices in every
 * tree): out_rows = [n][leaf_len], out_siblings = [n][log2(n_leaves) - cap_height][4]; either may be NULL                     */
int gl_tree_open_batch(gl_ctx* ctx, gl_handle tree, const uint64_t* leaf_indices, uint32_t n, uint64_t* out_rows,
                       uint64_t* out_siblings);
/* leaves[bitrev(index * step)] — PolynomialBatch::get_lde_values */
int gl_tree_get_lde_values(gl_ctx* ctx, gl_handle tree, uint64_t index, uint64_t step, uint64_t* out_row);
enum { GL_PART_COEFFS = 0, GL_PART_LEAVES = 1, GL_PART_DIGESTS = 2, GL_PART_CAP = 3 };
/* bulk device -> host copy of one part, same layouts as gl_commit's outputs */
int gl_tree_read(gl_ctx* ctx, gl_handle tree, int part, uint64_t* out);
int gl_tree_free(gl_ctx* ctx, gl_handle tree);

/* ---- FRI commit phase: fri_committed_trees  (plonky2 fri/prover.rs) ------------------------------------------
 * The Fiat–Shamir challenger stays on the host (upstream code, untouched); per layer the host calls
 *     gl_fri_commit_layer -> observes the cap, draws beta -> gl_fri_fold(beta)
 * coeffs / values: `len` extension elements each, interleaved [a0, a1]; values = coset_fft(coeffs, shift 7) in
 * natural order, exactly the two arguments upstream passes.                                                     */
int gl_fri_begin(gl_ctx* ctx, const uint64_t* coeffs_ext, const uint64_t* values_ext, uint64_t len,
                 uint32_t rate_bits, uint32_t cap_height, gl_handle* out_fri);
/* reverse_index_bits_in_place(values); leaves = chunks(2^arity_bits).flatten(); MerkleTree::new(leaves, cap_height) */
int gl_fri_commit_layer(gl_ctx* ctx, gl_handle fri, uint32_t arity_bits, uint64_t* out_leaves, uint64_t* out_digests,
                        uint64_t* out_cap, gl_handle* out_tree);
/* coeffs <- reduce_with_powers over chunks; shift <- shift^arity; values <- coset_fft(coeffs, shift) */
int gl_fri_fold(gl_ctx* ctx, gl_handle fri, const uint64_t beta[2]);
/* coeffs truncated to len >> rate_bits (final_poly); out_len in extension elements */
int gl_fri_final_poly(gl_ctx* ctx, gl_handle fri, uint64_t* out_coeffs_ext, uint64_t* out_len);
int gl_fri_end(gl_ctx* ctx, gl_handle fri);

/* ---- prove_openings, front half  (plonky2 fri/oracle.rs · PolynomialBatch::prove_openings) ----------------------
 * Builds the polynomial that goes into FRI from the device-resident coefficient matrices of earlier commits:
 *     final_poly = 0
 *     for every FriBatchInfo { point, polynomials }:                          (gl_openings_add_batch)
 *         F        = sum_j alpha^j * f_j                 ReducingFactor::reduce_polys_base (powers restart at alpha^0)
 *         quotient = (F(X) - F(point)) / (X - point)     divide_by_linear, then coeffs.push(ZERO)
 *         final_poly = final_poly * alpha^(number of polynomials of this batch) + quotient     shift_poly, +=
 *     lde_final_poly = final_poly.lde(rate_bits); lde_final_values = lde_final_poly.coset_fft(7)     (gl_openings_lde)
 * polynomial j of a batch is column columns[j] of the commit behind handle batches[j] (all commits of degree 2^log_n);
 * alpha, point: extension elements [a0, a1].  gl_openings_lde hands the result to the FRI commit phase as a gl_fri
 * handle (what gl_fri_begin would build from host arrays) without leaving the device.                                */
int gl_openings_begin(gl_ctx* ctx, uint32_t log_n, gl_handle* out_openings);
int gl_openings_add_batch(gl_ctx* ctx, gl_handle openings, const gl_handle* batches, const uint32_t* columns, uint32_t n_polys,
                          const uint64_t alpha[2], const uint64_t point[2], uint64_t* out_quotient_ext /* N*2 words or NULL */);
int gl_openings_final_poly(gl_ctx* ctx, gl_handle openings, uint64_t* out_coeffs_ext /* N*2 words */);
int gl_openings_lde(gl_ctx* ctx, gl_handle openings, uint32_t rate_bits, uint32_t cap_height, gl_handle* out_fri);
int gl_openings_end(gl_ctx* ctx, gl_handle openings);

/* ---- OpeningSet::new  (plonky2 plonk/proof.rs; the eval_commitment closure) ----------------------------------
 * Evaluates every polynomial of a committed batch at n_points extension points [a0, a1] (inputs may be non-canonical):
 * out_values = [n_points][leaf_len][2] words, canonical; out[p][j] = sum_k coeffs_j[k] * points[p]^k.
 * 1 <= n_points <= 2 (zeta; zeta and g*zeta for the Z commit).  The coefficient matrix never leaves the device.
 * A tree without coefficients (gl_merkle_new trees, gl_commit_multi shard trees) is refused with GL_ERR_INVALID.     */
int gl_batch_eval(gl_ctx* ctx, gl_handle batch, const uint64_t* points_ext, uint32_t n_points, uint64_t* out_values_ext);

/* read the current coefficients (len extension elements) / bit-reversed values of a gl_fri state (tests, debugging) */
int gl_fri_read(gl_ctx* ctx, gl_handle fri, uint64_t* out_coeffs_ext, uint64_t* out_values_bitrev_ext, uint64_t* out_len);

/* ---- gate constraints over the resident LDE rows, and witness rows (SURVEY §8f ranks 3-4) -------------------------------------
 * plonky2 plonk/prover.rs · compute_quotient_polys evaluates every gate's constraints at every point of the LDE coset and combines them
 * with powers of the challenges alpha_k (plonk/vanishing_poly.rs · evaluate_gate_constraints_base_batch + plonk_common.rs ·
 * reduce_with_powers).  The rows are already in HBM: a leaf row of the wires commit IS the wire vector at LDE point bitrev(row).
 * Gates implemented are the reference's own, whose source is in its tree:
 *   GL_GATE_POSEIDON2       /root/reference/src/common/poseidon2/poseidon2_gate.rs:233-310   135 wires, 123 constraints (param unused)
 *   GL_GATE_U32_ARITHMETIC  /root/reference/src/common/u32/gates/arithmetic_u32.rs:103-166    param = num_ops (3 at 135 wires / 80 routed):
 *                                                                                             38*num_ops wires, 36*num_ops constraints
 *   GL_GATE_U32_ADD_MANY    .../add_many_u32.rs:103-143        param = num_addends | num_ops << 8      (num_addends+21)*num_ops wires, 21*num_ops constraints
 *   GL_GATE_U32_SUBTRACTION .../subtraction_u32.rs:100-134     param = num_ops (<= 6)                   21*num_ops wires, 19*num_ops constraints
 *   GL_GATE_U32_RANGE_CHECK .../range_check_u32.rs:70-92       param = num_input_limbs (<= 7)           17*n wires, 17*n constraints
 *   GL_GATE_U32_INTERLEAVE  .../interleave_u32.rs:104-140      param = num_ops (<= 3)                   34*num_ops wires and constraints
 *   GL_GATE_UNINTERLEAVE_TO_U32 / _TO_B32  .../uninterleave_to_u32.rs:91-134, uninterleave_to_b32.rs:115-168   param = num_ops (<= 2)   67*num_ops each
 *   GL_GATE_COMPARISON      .../comparison.rs:112-190          param = num_bits | num_chunks << 8      5*num_chunks + chunk_bits + 5 wires, + 6 constraints
 * and plonky2's core gates (plonky2 @ 3de92d9 gates/{noop,constant,public_input,arithmetic_base,base_sum}.rs; upstream source not in
 * the reference tree: restated, parity unpinned):
 *   GL_GATE_NOOP            NoopGate                           param 0                                  0 wires, 0 constraints, 0 constants
 *   GL_GATE_CONSTANT        ConstantGate                       param = num_consts (1..8)                n wires, n constraints, n constants
 *   GL_GATE_PUBLIC_INPUT    PublicInputGate                    param 0                                  4 wires, 4 constraints, 0 constants
 *   GL_GATE_ARITHMETIC      ArithmeticGate (base)              param = num_ops (1..33; 20 at 80 routed)  4*n wires, n constraints, 2 constants
 *   GL_GATE_BASE_SUM        BaseSumGate<B>                     param = num_limbs | B << 8 (B 2..16)      1+n wires, 1+n constraints, 0 constants
 * and three more base-field gates of plonky2 @ 3de92d9 (gates/{poseidon,exponentiation,random_access}.rs; restated, parity unpinned):
 *   GL_GATE_POSEIDON        PoseidonGate                       param 0                                  135 wires, 123 constraints, 0 constants
 *                           (Poseidon2Gate's wire layout; the permutation is the leaf hash's plonky2 Poseidon)
 *   GL_GATE_EXPONENTIATION  ExponentiationGate                 param = num_power_bits (1..66; 66 at 135 wires / 80 routed)
 *                                                              2+2n wires, n+1 constraints, 0 constants
 *   GL_GATE_RANDOM_ACCESS   RandomAccessGate                   param = bits | num_copies << 8 | num_extra_constants << 16
 *                           (bits 1..6, v = 2^bits, (2+v+bits)*num_copies + num_extra_constants <= 135 wires)
 *                                                              (bits+2)*num_copies + num_extra_constants constraints, num_extra_constants constants
 * Kind 14 is not assigned: it stays an unknown kind, as it was before these three gates existed.
 * gl_quotient_add_gate:  acc[k][row] += filter(row) * sum_i alphas[k]^(constraint_offset + i) * constraint_i(wires(row)),  k < n_challenges
 * (alphas are BASE-field challenges, as upstream; filter(row) = column filter_col of the batch filter_batch at the same row, or 1 when
 * filter_batch == 0).  gl_quotient_read: [n_challenges][R] words, row order = the leaves' (bit-reversed).
 * gl_gate_eval_rows and gl_quotient_add_gate refuse the gates that read gate constants or the public-inputs hash (CONSTANT, ARITHMETIC,
 * PUBLIC_INPUT, and RANDOM_ACCESS with extra constants): those go through gl_gate_eval_rows_with_constants and gl_quotient_add_gates. */
enum { GL_GATE_POSEIDON2 = 0, GL_GATE_U32_ARITHMETIC = 1, GL_GATE_U32_ADD_MANY = 2, GL_GATE_U32_SUBTRACTION = 3, GL_GATE_U32_RANGE_CHECK = 4,
       GL_GATE_U32_INTERLEAVE = 5, GL_GATE_UNINTERLEAVE_TO_U32 = 6, GL_GATE_UNINTERLEAVE_TO_B32 = 7, GL_GATE_COMPARISON = 8, GL_GATE_NOOP = 9,
       GL_GATE_CONSTANT = 10, GL_GATE_PUBLIC_INPUT = 11, GL_GATE_ARITHMETIC = 12, GL_GATE_BASE_SUM = 13, GL_GATE_POSEIDON = 15,
       GL_GATE_EXPONENTIATION = 16, GL_GATE_RANDOM_ACCESS = 17 };
int gl_gate_num_wires(int kind, uint32_t param);
int gl_gate_num_constraints(int kind, uint32_t param);
/* Gate::num_constants: the gate constants a gate reads (-1 for a bad kind or parameter) */
int gl_gate_num_constants(int kind, uint32_t param);
/* every constraint value of every row, uncombined (host rows [n_rows][num_wires] -> out [n_rows][num_constraints]); tests, debugging */
int gl_gate_eval_rows(gl_ctx* ctx, int kind, uint32_t param, const uint64_t* rows, uint64_t n_rows, uint64_t* out);
/* gl_gate_eval_rows for every kind, with the gate constants of each row: consts [n_rows][gl_gate_num_constants] (NULL if that is 0) */
int gl_gate_eval_rows_with_constants(gl_ctx* ctx, int kind, uint32_t param, const uint64_t* rows, const uint64_t* consts,
                                     const uint64_t public_inputs_hash[4], uint64_t n_rows, uint64_t* out);
int gl_quotient_begin(gl_ctx* ctx, gl_handle wires_batch, uint32_t n_challenges, gl_handle* out_quotient);
int gl_quotient_add_gate(gl_ctx* ctx, gl_handle quotient, int kind, uint32_t param, const uint64_t* alphas, uint32_t constraint_offset,
                         gl_handle filter_batch, uint32_t filter_col);
/* plonky2 plonk/vanishing_poly.rs · evaluate_gate_constraints_base_batch over the resident LDE rows (restated, parity unpinned).
 * Gate i of CommonCircuitData::gates is (kinds[i], params[i]); SelectorsInfo is selector_indices[n_gates] and groups[2 * num_selectors]
 * ([start, end) pairs).  constants_sigmas: commit #0 — selectors, lookup selectors and gate constants in columns [0, num_constants), the
 * sigmas after; it shares the wires batch's rows, degree and rate_bits.  For every gate with constraints, one launch:
 *     s = constants_sigmas[row][selector_indices[i]],  f_i = prod_{j in group, j != i} (j - s) * (num_selectors > 1 ? 2^32 - 1 - s : 1)
 *     acc[k][row] += f_i * sum_c alphas[k]^(constraint_offset + c) * c_i,c(row)
 * with gate constant j = constants_sigmas[row][num_selectors + num_lookup_selectors + j] (gates/gate.rs · compute_filter,
 * eval_filtered_base_batch).  Every gate is validated before the first launch; a refused call leaves the accumulator unchanged. */
int gl_quotient_add_gates(gl_ctx* ctx, gl_handle quotient, const int* kinds, const uint32_t* params, uint32_t n_gates,
                          const uint32_t* selector_indices, const uint32_t* groups, uint32_t num_selectors, uint32_t num_lookup_selectors,
                          gl_handle constants_sigmas, uint32_t num_constants, const uint64_t public_inputs_hash[4], const uint64_t* alphas,
                          uint32_t constraint_offset);
/* the permutation-argument terms of eval_vanishing_poly_base_batch (plonk/vanishing_poly.rs; restated, parity unpinned): for every challenge i
 * L_0(x)(Z_i(x) - 1), then check_partial_products of every challenge — vanishing_terms[0 .. n_ch*(1 + n_chunks)), each alpha_k reducing the
 * whole list; gate constraints follow from constraint_offset = n_ch * (1 + n_chunks).  sigmas_batch: the constants+sigmas commit, the sigma
 * polynomials at columns [sigma_col0, sigma_col0 + n_routed); zs_batch: the commit of gl_partial_products' columns (Z first); all three
 * batches share the wires batch's degree and rate_bits.                                                                                 */
int gl_quotient_add_permutation(gl_ctx* ctx, gl_handle quotient, gl_handle sigmas_batch, uint32_t sigma_col0, gl_handle zs_batch,
                                uint32_t n_routed, uint32_t degree, const uint64_t* k_is, const uint64_t* betas, const uint64_t* gammas,
                                const uint64_t* alphas);
int gl_quotient_read(gl_ctx* ctx, gl_handle quotient, uint64_t* out);
/* the tail of compute_quotient_polys and the quotient commit of prove() (plonky2 plonk/prover.rs), without leaving the device:
 * acc_k / Z_H on the coset (ZeroPolyOnCoset::eval_inverse), coset_ifft(7) to coefficients (degree < 2^rate_bits * N), split into
 * 2^rate_bits chunks of N coefficients each (quotient_degree_factor = 2^rate_bits, the reference's configuration), and
 * PolynomialBatch::from_coeffs of the n_challenges * 2^rate_bits chunk polynomials (challenge-major).  out_cap: 2^cap_height * 4 words;
 * out_batch: the committed batch (coefficients, leaves, digests resident), as from gl_commit.  Restated from upstream (parity unpinned).  */
int gl_quotient_commit(gl_ctx* ctx, gl_handle quotient, uint32_t cap_height, uint64_t* out_cap, gl_handle* out_batch);
int gl_quotient_end(gl_ctx* ctx, gl_handle quotient);
/* CUDA-event milliseconds of the last gl_quotient_add_gate / gl_poseidon2_gate_witness / gl_poseidon_gate_witness kernel on this context (gl_quotient_add_gates:
 * from its first launch to its last; 0 when it launched nothing) */
int gl_ctx_aux_ms(gl_ctx* ctx, float* out_ms);
/* witness generation for Poseidon2Gate rows (poseidon2_gate.rs:447-523 · Poseidon2Generator::run_once): inputs [n][13] = the 12 state
 * inputs + the swap flag of each row -> out_rows [n][135], every wire of the row (deltas, S-box inputs of all rounds, outputs)        */
int gl_poseidon2_gate_witness(gl_ctx* ctx, const uint64_t* inputs, uint64_t n, uint64_t* out_rows);
/* witness generation for plonky2's PoseidonGate rows (gates/poseidon.rs · PoseidonGenerator::run_once; restated, parity unpinned): the
 * same shape as gl_poseidon2_gate_witness — inputs [n][13] -> out_rows [n][135], every wire written, canonical; swap applied when it is 1 */
int gl_poseidon_gate_witness(gl_ctx* ctx, const uint64_t* inputs, uint64_t n, uint64_t* out_rows);

/* ---- permutation argument: partial products and Z (SURVEY §8f rank 4) --------------------------------------------------------
 * plonky2 plonk/prover.rs · all_wires_permutation_partial_products (+ the "Z first" reordering prove() applies before committing):
 * per challenge k and row i (x_i = w_N^i):  q_ic = prod_{j in chunk c of `degree` routed wires} (wire_ij + beta_k k_j x_i + gamma_k) /
 * (wire_ij + beta_k sigma_ij + gamma_k); a running product over (i, c) from Z(x_0) = 1 gives the partial products and Z(x_{i+1}).
 * wire_cols / sigma_cols: n_routed host pointers each, N = 2^log_n words (witness wire values; sigma polynomial VALUES on the subgroup,
 * i.e. prover_data.sigmas transposed); k_is: the n_routed coset shifts (get_unique_coset_shifts: 7^j).
 * out_cols: [(n_challenges * n_chunks)][N] words, n_chunks = ceil(n_routed / degree): first the Z polynomial of every challenge, then
 * the n_chunks - 1 partial products of challenge 0, of challenge 1, ... — the column order of the Z/partial-products commit.
 * Upstream source is not in /root/reference: restated (parity unpinned), see plonky2.5_b200/csrc/permutation.cuh.                     */
int gl_partial_products(gl_ctx* ctx, const uint64_t* const* wire_cols, const uint64_t* const* sigma_cols, uint32_t n_routed, uint32_t log_n,
                        const uint64_t* k_is, const uint64_t* betas, const uint64_t* gammas, uint32_t n_challenges, uint32_t degree,
                        uint64_t* out_cols);

/* ---- FRI proof of work: fri_proof_of_work  (plonky2 fri/prover.rs) ---------------------------------------------
 * sponge_state / input_buffer: the caller's Challenger fields (sponge_state, pending input_buffer, n_inputs < 8).
 * Finds the SMALLEST canonical w such that, with the pending inputs written into the state and w in the next input
 * lane, permute(state)[7] has >= min_leading_zeros leading zero bits (= what the serial `find` of the reference build,
 * plonky2 `parallel` off, returns; deterministic).  The caller then observes w and draws the response as upstream. */
int gl_fri_pow(gl_ctx* ctx, const uint64_t sponge_state[12], const uint64_t* input_buffer, uint32_t n_inputs,
               uint32_t min_leading_zeros, uint64_t* out_witness);

/* ---- Poseidon permutation batch (plonky2 hash/poseidon.rs · PoseidonPermutation::permute) ---------------------
 * states: n x 12 words, permuted in place, canonical on return.  Used by the host-side Challenger mirror.       */
int gl_poseidon_permute(gl_ctx* ctx, uint64_t* states, uint64_t n);

/* The Challenger's duplexing loop over n_groups FULL groups of 8 observed elements (iop/challenger.rs · observe_elements): for each group,
 * state[0..8) <- group; state <- permute(state).  One launch and one round trip per call (a Merkle cap of 16 hashes = 8 groups), state
 * canonical on return.  The host-side Challenger keeps its input/output buffers and calls this for the full groups.                   */
int gl_poseidon_absorb(gl_ctx* ctx, uint64_t state[12], const uint64_t* groups, uint32_t n_groups);

/* ---- device-pointer stage API (inputs/outputs already in HBM; multi-GPU host code and benchmarks) ------------- */
/* whole commit from a device-resident column-major matrix d_cols[n_cols][2^log_n] (col_stride words apart) */
int gl_dev_commit(gl_ctx* ctx, const uint64_t* d_cols, uint64_t col_stride, uint32_t n_cols, uint32_t log_n,
                  uint32_t rate_bits, uint32_t cap_height, int input_is_coeffs, uint64_t* out_cap, gl_handle* out_batch);
/* stage 1 of the sharded commit: iNTT + coset LDE of a column shard; d_out_rows = [R][out_pitch] row-major
 * (out_pitch multiple of 4), rows in bit-reversed LDE order; d_out_coeffs = [N][out_pitch] or NULL              */
int gl_dev_lde(gl_ctx* ctx, const uint64_t* d_cols, uint64_t col_stride, uint32_t n_cols, uint32_t log_n,
               uint32_t rate_bits, int input_is_coeffs, uint64_t* d_out_rows, uint32_t out_pitch,
               uint64_t* d_out_coeffs);
/* stage 1 fused with the column->row exchange (one process per GPU, NVLink peer memory): like gl_dev_lde, but every coset's
 * rows go to the leaf buffer of the rank that owns them.  A coset whose rows all belong to this rank (its buffer is one
 * allocated by gl_dev_ipc_alloc on ctx) is stored there by the last NTT pass itself; every other coset is evaluated into a
 * local buffer and shipped by the copy engines, one strided peer copy per owner, while the next coset's NTT runs.
 * Global leaf row i lives in peer_leaves[i / (R/n_peers)] at row i % (R/n_peers), columns [col_off, col_off+n_cols) of
 * a [R/n_peers][leaf_pitch] matrix.  peer_leaves: HOST array of n_peers device pointers (own buffer + buffers mapped
 * with gl_dev_ipc_open).  The caller synchronises the ranks (barrier) before hashing.  The 2^rate_bits cosets are
 * processed in the order first_coset, first_coset+1, ... (mod 2^rate_bits): ranks that start at different cosets store
 * to different owners at any one time instead of all converging on one GPU's NVLink ingress.                        */
int gl_dev_lde_scatter(gl_ctx* ctx, const uint64_t* d_cols, uint64_t col_stride, uint32_t n_cols, uint32_t log_n,
                       uint32_t rate_bits, int input_is_coeffs, uint64_t* const* peer_leaves, uint32_t n_peers,
                       uint32_t leaf_pitch, uint32_t col_off, uint64_t* d_out_coeffs, uint32_t coeff_pitch,
                       uint32_t first_coset);
/* the same with HOST columns (cols[j] = N words, as gl_commit): the shard is copied in growing chunks on a copy stream while
 * the NTTs of the previous chunk run, so only the first 8-column copy is exposed                                        */
int gl_lde_scatter(gl_ctx* ctx, const uint64_t* const* cols, uint32_t n_cols, uint32_t log_n, uint32_t rate_bits,
                   int input_is_coeffs, uint64_t* const* peer_leaves, uint32_t n_peers, uint32_t leaf_pitch, uint32_t col_off,
                   uint64_t* d_out_coeffs, uint32_t coeff_pitch, uint32_t first_coset);
/* ---- coset-sharded commit (one process per GPU; the default multi-GPU plan when n_ranks <= 2^rate_bits) --------------------------------
 * Leaf rows are stored in bit-reversed LDE order, so the contiguous leaf range a rank owns is a set of whole LDE cosets (SURVEY F10).
 * Instead of exchanging LDE OUTPUT column->row (R x C words in 8C/G-byte pieces), the ranks exchange COEFFICIENTS: every rank runs the
 * iNTT of its column shard (gl_dev_intt), pulls the other ranks' coefficient blocks — whole contiguous [N][pitch] buffers, one large
 * NVLink copy each, overlapped with the NTTs of the blocks that have already arrived — and evaluates only ITS OWN cosets for ALL columns,
 * writing its leaf rows in place (gl_dev_lde_own_cosets).  Same bytes on the wire per rank (8 C N (G-1)/G), no strided shipment, no exposed
 * tail, LDE work perfectly balanced.
 * gl_dev_intt: d_out_coeffs [N][coeff_pitch] <- iNTT (or canonical copy if input_is_coeffs) of the n_cols device columns.
 * gl_dev_lde_own_cosets: peer_coeffs[q] = rank q's coefficient block (own buffer for q == self, CUDA-IPC mapping otherwise), with
 * pitches[q], col_counts[q], col_offsets[q]; d_stage[q] = local staging for rank q's block (ignored for q == self);
 * leaf blocks [self*2^rate_bits/n_peers, (self+1)*2^rate_bits/n_peers) are written to d_leaves [rows_per_rank][leaf_pitch].
 * The caller synchronises the ranks between the two calls (every block complete) — see plonky2.5_b200/sharded.py.                   */
int gl_dev_intt(gl_ctx* ctx, const uint64_t* d_cols, uint64_t col_stride, uint32_t n_cols, uint32_t log_n, int input_is_coeffs,
                uint64_t* d_out_coeffs, uint32_t coeff_pitch);
/* gl_dev_intt with HOST columns (cols[j] = N words): chunked host->device copies overlapped with the transposes / iNTTs of the previous chunk */
int gl_intt_host(gl_ctx* ctx, const uint64_t* const* cols, uint32_t n_cols, uint32_t log_n, int input_is_coeffs, uint64_t* d_out_coeffs,
                 uint32_t coeff_pitch);
int gl_dev_lde_own_cosets(gl_ctx* ctx, uint64_t* const* peer_coeffs, uint64_t* const* d_stage, const uint32_t* pitches,
                          const uint32_t* col_counts, const uint32_t* col_offsets, uint32_t n_peers, uint32_t self, uint32_t log_n,
                          uint32_t rate_bits, uint64_t* d_leaves, uint32_t leaf_pitch);

/* ---- the coset-sharded commit, STREAMED from host columns (one process per GPU; what a multi-GPU PolynomialBatch::from_values pays) ----
 * With host inputs the plan above cannot start before every rank's whole shard has crossed PCIe.  Here the batch is cut into WAVES of
 * n_peers * group_width consecutive columns; in wave w rank q owns the group_width columns [gw*(w*G+q), gw*(w*G+q+1)) (cyclic deal).
 * Per wave every rank copies its group host->device, runs its iNTT on a high-priority stream and publishes a ticket to every peer
 * (csrc/peer_sync.cuh: release stores into the peers' flag arrays, no host round trip, no collective); the peers' copy engines pull the
 * group over NVLink as soon as the ticket shows; the rank then evaluates ITS OWN cosets of the wave's G groups and ABSORBS the wave's
 * columns into the leaf sponge (the overwrite-mode sponge consumes a leaf strictly left to right).  Copies, pulls and NTTs of wave w+1
 * run while wave w is hashed, so only the first wave's copy is exposed; the tree above the digests follows the last wave.
 * Same permutations in the same order as the one-GPU commit => the same digests and cap, bit for bit.
 *
 * Buffers: every rank exports ONE buffer (gl_dev_ipc_alloc, zero-filled) of `exported_words` = n_waves * N * gw coefficient words
 * followed by n_peers * n_waves ticket words; peer_bufs[q] = rank q's (own pointer for q == self).  d_stage = `stage_words` local words
 * (the pulled groups), d_leaves = [rows_per_rank][leaf_pitch], d_digests as gl_dev_merkle.  own_cols = the rank's columns in wave order
 * (gl_stream_plan_sizes reports how many).  epoch: the number of earlier calls on these buffers — the same on every rank.  The caller must
 * put a collective (the cap all-gather) between two calls, as for gl_dev_lde_own_cosets.  A peer that does not publish within
 * GL_PEER_TIMEOUT_MS (default 20000) makes the call fail with GL_ERR_CUDA instead of hanging. */
typedef struct {
    uint32_t n_cols;       /* C: columns of the WHOLE batch */
    uint32_t log_n;
    uint32_t rate_bits;
    uint32_t cap_height;   /* of the rank's own leaf range (global cap height - log2 n_peers) */
    uint32_t n_peers;      /* G, a power of two <= 2^rate_bits */
    uint32_t self;
    uint32_t group_width;  /* gw: 4 or 8; n_peers * gw must be a multiple of 8 (the sponge rate) */
    uint32_t leaf_pitch;   /* words per device leaf row, multiple of 8, >= round_up(C, 8) */
    uint64_t epoch;
} gl_stream_plan_t;
int gl_stream_plan_sizes(const gl_stream_plan_t* plan, uint64_t* exported_words, uint64_t* stage_words, uint32_t* n_waves,
                         uint32_t* n_own_cols);
int gl_commit_coset_stream(gl_ctx* ctx, const gl_stream_plan_t* plan, const uint64_t* const* own_cols, int input_is_coeffs,
                           uint64_t* const* peer_bufs, uint64_t* d_stage, uint64_t* d_leaves, uint64_t* d_digests, uint64_t* out_cap);

/* CUDA IPC plumbing for the above: export a device buffer (64-byte handle) / map a peer's / unmap / free */
int gl_dev_ipc_alloc(gl_ctx* ctx, uint64_t words, uint64_t** out_ptr, uint8_t out_handle[64]);
int gl_dev_ipc_open(gl_ctx* ctx, const uint8_t handle[64], uint64_t** out_ptr);
int gl_dev_ipc_close(gl_ctx* ctx, uint64_t* ptr);
int gl_dev_ipc_free(gl_ctx* ctx, uint64_t* ptr);
/* copy the first src_cols columns of a received [n_rows][src_pitch] block into columns
 * [dst_col_off, dst_col_off+src_cols) of [n_rows][dst_pitch] (canonicalising) */
int gl_dev_repack(gl_ctx* ctx, const uint64_t* d_src, uint32_t src_pitch, uint32_t src_cols, uint64_t n_rows, uint64_t* d_dst,
                  uint32_t dst_pitch, uint32_t dst_col_off);
/* stage 3: Merkle subtrees over device rows [n_leaves][pitch]; d_digests 2*(n_leaves-2^cap_height)*4 words (device),
 * out_cap host 2^cap_height*4 */
int gl_dev_merkle(gl_ctx* ctx, const uint64_t* d_leaves, uint64_t n_leaves, uint32_t leaf_len, uint32_t pitch,
                  uint32_t cap_height, uint64_t* d_digests, uint64_t* out_cap);

/* plain device memory + copies for hosts without a CUDA binding of their own (tests, the C++ tools): words are uint64_t */
int gl_dev_alloc(gl_ctx* ctx, uint64_t words, uint64_t** out_ptr);
int gl_dev_free(gl_ctx* ctx, uint64_t* ptr);
int gl_dev_upload(gl_ctx* ctx, const uint64_t* host_src, uint64_t* d_dst, uint64_t words);
int gl_dev_download(gl_ctx* ctx, const uint64_t* d_src, uint64_t* host_dst, uint64_t words);

/* ---- instrumentation ---------------------------------------------------------------------------------------- */
enum {
    GL_STAGE_H2D = 0, GL_STAGE_TRANSPOSE = 1, GL_STAGE_INTT = 2, GL_STAGE_LDE = 3, GL_STAGE_LEAF_HASH = 4,
    GL_STAGE_TREE = 5, GL_STAGE_D2H = 6, GL_N_STAGES = 7
};
/* CUDA-event milliseconds of the stages of the last gl_commit / gl_dev_commit on this context (timed on the
 * context's stream); kernel launch counts of that call in out_launches[GL_N_STAGES] (may be NULL). */
int gl_ctx_stage_times(gl_ctx* ctx, float* out_ms, uint32_t* out_launches);
/* integer-pipe calibration (K7): runs `iters` dependent-chain iterations of {0: IMAD.WIDE.U32, 1: IADD3, 2: mixed,
 * 3: Goldilocks modmul, 4: Poseidon permutation} on every SM, returns operations per second in *out_ops_per_s */
int gl_microbench(gl_ctx* ctx, int which, uint32_t iters, double* out_ops_per_s);

/* element-wise field primitives exactly as the kernels use them (carry-logic unit tests on adversarial words).
 * out[i] = op(a[i], b[i]) canonicalised, or the raw 64-bit representative when GL_FOP_RAW is or-ed in.             */
enum {
    GL_FOP_MUL = 0, GL_FOP_ADD_ANY = 1, GL_FOP_SUB_ANY = 2, GL_FOP_MUL_2_24 = 3, GL_FOP_MUL_2_48 = 4, GL_FOP_MUL_2_72 = 5,
    GL_FOP_SBOX7 = 6, GL_FOP_ADD_ANY_C = 7, GL_FOP_RAW = 0x100
};
int gl_field_op(gl_ctx* ctx, int op, const uint64_t* a, const uint64_t* b, uint64_t* out, uint64_t n);

/* pinned host memory for benchmarks / shims that want fast PCIe copies */
void* gl_host_alloc(size_t bytes);
void gl_host_free(void* p);

#ifdef __cplusplus
}
#endif
#endif /* GL_COMMIT_H */
