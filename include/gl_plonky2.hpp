/*
 * gl_plonky2.hpp — C++17 host-side mirror of the plonky2 operator interface for the commitment hot path, header-only,
 * on top of the C ABI in gl_commit.h.
 *
 * The reference (/root/reference, crate plonky2_5) is Rust and reaches this path through `builder.build::<C>()`
 * (src/p3/mod.rs:250) and `data.prove(pw)` (src/p3/mod.rs:260), which land in its pinned dependency
 * plonky2 @ 3de92d9ed1721cec133e4e1e1b3ec7facb756ccf (Cargo.toml:15-19).  No Rust toolchain exists in this image, so
 * the compiled-language host layer a maintainer would write in Rust (INTEGRATION.md) is provided here in C++ with the
 * SAME item names, argument order and meaning, and error behaviour as upstream:
 *
 *     plonky2 fri/oracle.rs          PolynomialBatch::{from_values, from_coeffs, get_lde_values, prove_openings}
 *     plonky2 hash/merkle_tree.rs    MerkleTree::{new, get, prove}, MerkleCap;  hash/merkle_proofs.rs  MerkleProof
 *     plonky2 fri/prover.rs          fri_proof, fri_committed_trees, fri_proof_of_work, fri_prover_query_rounds
 *     plonky2 fri/{mod,structure,proof}.rs   FriConfig, FriParams, FriInstanceInfo, FriBatchInfo, FriPolynomialInfo,
 *                                    FriProof, FriQueryRound, FriInitialTreeProof, FriQueryStep
 *     plonky2 iop/challenger.rs      Challenger<GoldilocksField, PoseidonHash>, observe_openings
 *     plonky2 plonk/proof.rs         OpeningSet::{new, to_fri_openings};  fri/structure.rs  FriOpenings, FriOpeningBatch
 *
 * (`new` is a C++ keyword: MerkleTree::new_.)  Upstream functions are infallible and `assert!`-panic on misuse; here a
 * violated upstream assert throws plonky2::Panic carrying the upstream message, any other failure (no CUDA device,
 * CUDA error, out of memory) throws plonky2::GlError.  There is NO CPU path in this file: every permutation, NTT and hash
 * runs in libgl_commit on the GPU, and constructing a Context without a CUDA device throws.
 *
 * Field elements are `uint64_t` words (GoldilocksField is #[repr(transparent)] struct(pub u64)); extension elements are
 * two words [a0, a1] of F_p[X]/(X^2 - 7) (reference: src/p3/extension.rs:458-470).  Inputs may be non-canonical, outputs
 * are canonical.  Trees and batches stay resident in HBM; `leaves()`, `digests()` and `polynomials()` copy back on demand.
 */
#ifndef GL_PLONKY2_HPP
#define GL_PLONKY2_HPP

#include <array>
#include <cstdint>
#include <memory>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "gl_commit.h"

namespace plonky2 {

using F = uint64_t;                         /* GoldilocksField */
using Ext = std::array<uint64_t, 2>;        /* QuadraticExtension<GoldilocksField>: a0 + a1 X, X^2 = 7 */
constexpr uint64_t ORDER = 0xFFFFFFFF00000001ULL;
constexpr size_t SPONGE_RATE = 8, SPONGE_WIDTH = 12;

/* what an upstream `assert!` / `panic!` becomes on this side of the boundary */
struct Panic : std::logic_error { using std::logic_error::logic_error; };
/* CUDA / device / allocation failures of libgl_commit (there is no CPU fallback to hide them) */
struct GlError : std::runtime_error {
    int code;
    GlError(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};

struct TimingTree {};     /* accepted and ignored, as in the reference build (upstream's timing tree is compiled out) */
struct FftRootTable {};   /* the device keeps its own twiddle tables; the argument is accepted for signature parity */

struct PolynomialValues { std::vector<F> values; size_t len() const { return values.size(); } };
struct PolynomialCoeffs { std::vector<F> coeffs; size_t len() const { return coeffs.size(); } };
struct PolynomialCoeffsExt { std::vector<Ext> coeffs; size_t len() const { return coeffs.size(); } };
struct PolynomialValuesExt { std::vector<Ext> values; size_t len() const { return values.size(); } };

struct HashOut {
    std::array<F, 4> elements{};
    bool operator==(const HashOut& o) const { return elements == o.elements; }
    bool operator!=(const HashOut& o) const { return !(*this == o); }
};
static_assert(sizeof(HashOut) == 32, "HashOut must be 4 packed words (gl_commit.h layouts)");
static_assert(sizeof(Ext) == 16, "extension elements must be 2 packed words");

struct MerkleCap {
    std::vector<HashOut> hashes;            /* upstream: MerkleCap(pub Vec<H::Hash>) */
    size_t len() const { return hashes.size(); }
    size_t height() const { size_t h = 0; while ((size_t(1) << h) < hashes.size()) h++; return h; }
    std::vector<F> flatten() const {
        std::vector<F> v;
        v.reserve(4 * hashes.size());
        for (const auto& h : hashes) v.insert(v.end(), h.elements.begin(), h.elements.end());
        return v;
    }
};

struct MerkleProof { std::vector<HashOut> siblings; size_t len() const { return siblings.size(); } };

/* plonky2 fri/structure.rs · FriOpeningBatch { values }, FriOpenings { batches } */
struct FriOpeningBatch { std::vector<Ext> values; };
struct FriOpenings { std::vector<FriOpeningBatch> batches; };

/* ------------------------------------------------------------------------------------------------ Context */
/* One CUDA device + stream + cached twiddle tables (gl_ctx).  Calls on one Context are serialised by the library;
 * use one Context per prover thread (Context::thread_default()). */
class Context {
public:
    explicit Context(int device = 0) {
        int rc = gl_ctx_create(&ctx_, device);
        if (rc != GL_OK) {
            ctx_ = nullptr;
            throw GlError(rc, std::string("gl_ctx_create(device=") + std::to_string(device) + ") failed: " + gl_strerror(rc) +
                                  " (libgl_commit has no CPU fallback; a CUDA device is required)");
        }
    }
    ~Context() { if (ctx_) gl_ctx_destroy(ctx_); }
    Context(const Context&) = delete;
    Context& operator=(const Context&) = delete;

    gl_ctx* raw() const { return ctx_; }

    /* status code -> the exception the upstream panic / failure corresponds to */
    void check(int rc) const {
        if (rc == GL_OK) return;
        std::string text = std::string(gl_strerror(rc)) + ": " + gl_ctx_last_error(ctx_);
        if (rc == GL_ERR_INVALID) throw Panic(text);
        throw GlError(rc, text);
    }

    /* PoseidonPermutation::permute on `n` states of 12 words, in place, on the device */
    void poseidon_permute(uint64_t* states, uint64_t n) const { check(gl_poseidon_permute(ctx_, states, n)); }

    /* the context the upstream-signature entry points use when none is passed: one per calling thread */
    static Context& thread_default() {
        thread_local std::unique_ptr<Context> c;
        if (!c) c = std::make_unique<Context>(0);
        return *c;
    }

private:
    gl_ctx* ctx_ = nullptr;
};

inline Context& ctx_or_default(Context* c) { return c ? *c : Context::thread_default(); }

/* ------------------------------------------------------------------------------------------------ MerkleTree */
/* plonky2 hash/merkle_tree.rs · MerkleTree<GoldilocksField, PoseidonHash> { leaves, digests, cap }.  The leaves and
 * digests live in HBM behind a handle; `cap` is always on the host. */
class MerkleTree {
public:
    MerkleCap cap;

    MerkleTree() = default;
    MerkleTree(Context& ctx, gl_handle h, MerkleCap c) : cap(std::move(c)), ctx_(&ctx), h_(h) {
        ctx.check(gl_tree_info(ctx.raw(), h, &info_));
    }
    MerkleTree(MerkleTree&& o) noexcept { *this = std::move(o); }
    MerkleTree& operator=(MerkleTree&& o) noexcept {
        if (this != &o) {
            release();
            cap = std::move(o.cap); ctx_ = o.ctx_; h_ = o.h_; info_ = o.info_;
            leaves_ = std::move(o.leaves_); digests_ = std::move(o.digests_);
            have_leaves_ = o.have_leaves_; have_digests_ = o.have_digests_;
            o.h_ = 0; o.ctx_ = nullptr;
        }
        return *this;
    }
    MerkleTree(const MerkleTree&) = delete;
    MerkleTree& operator=(const MerkleTree&) = delete;
    ~MerkleTree() { release(); }

    /* MerkleTree::new(leaves: Vec<Vec<F>>, cap_height) */
    static MerkleTree new_(const std::vector<std::vector<F>>& leaves, size_t cap_height, Context* ctx = nullptr) {
        if (leaves.empty()) throw Panic("MerkleTree::new: no leaves");
        const size_t n = leaves.size(), len = leaves[0].size();
        std::vector<F> flat;
        flat.reserve(n * len);
        for (const auto& l : leaves) {
            if (l.size() != len) throw Panic("MerkleTree::new: leaves of unequal length");
            flat.insert(flat.end(), l.begin(), l.end());
        }
        return from_flat(flat.data(), n, len, cap_height, ctx);
    }
    /* the same over packed row-major leaves (no Vec<Vec<F>> allocations) */
    static MerkleTree from_flat(const F* leaves, size_t n_leaves, size_t leaf_len, size_t cap_height, Context* ctx = nullptr) {
        Context& c = ctx_or_default(ctx);
        /* upstream's assert, checked before the cap is sized by 2^cap_height */
        if (cap_height >= 64 || n_leaves == 0 || (size_t(1) << cap_height) > n_leaves)
            throw Panic("cap_height=" + std::to_string(cap_height) + " should be at most log2(leaves.len())");
        MerkleCap cap;
        cap.hashes.resize(size_t(1) << cap_height);
        gl_handle h = 0;
        c.check(gl_merkle_new(c.raw(), leaves, n_leaves, uint32_t(leaf_len), uint32_t(cap_height), nullptr,
                              cap.hashes[0].elements.data(), &h));
        return MerkleTree(c, h, std::move(cap));
    }

    size_t n_leaves() const { return size_t(info_.n_leaves); }
    size_t leaf_len() const { return info_.leaf_len; }
    size_t cap_height() const { return info_.cap_height; }
    size_t degree_log() const { return info_.degree_log; }
    size_t rate_bits() const { return info_.rate_bits; }
    size_t depth() const { size_t d = 0; while ((size_t(1) << d) < n_leaves()) d++; return d - cap_height(); }
    gl_handle handle() const { return h_; }
    Context& context() const { return *ctx_; }

    /* MerkleTree::get(i) */
    std::vector<F> get(size_t i) const {
        std::vector<F> row(leaf_len());
        ctx_->check(gl_tree_get(ctx_->raw(), h_, i, row.data()));
        return row;
    }
    /* MerkleTree::prove(leaf_index): siblings bottom-up up to (not including) the cap */
    MerkleProof prove(size_t leaf_index) const {
        MerkleProof p;
        p.siblings.resize(depth());
        ctx_->check(gl_tree_prove(ctx_->raw(), h_, leaf_index, p.siblings.empty() ? nullptr : p.siblings[0].elements.data()));
        return p;
    }
    /* (get(i), prove(i)) for every i of `indices` in one device round trip */
    std::vector<std::pair<std::vector<F>, MerkleProof>> open_batch(const std::vector<uint64_t>& indices) const {
        const size_t n = indices.size(), d = depth(), ll = leaf_len();
        std::vector<F> rows(n * ll);
        std::vector<HashOut> sib(n * d);
        ctx_->check(gl_tree_open_batch(ctx_->raw(), h_, n ? indices.data() : nullptr, uint32_t(n), rows.empty() ? nullptr : rows.data(),
                                       sib.empty() ? nullptr : sib[0].elements.data()));
        std::vector<std::pair<std::vector<F>, MerkleProof>> out(n);
        for (size_t q = 0; q < n; q++) {
            out[q].first.assign(rows.begin() + q * ll, rows.begin() + (q + 1) * ll);
            out[q].second.siblings.assign(sib.begin() + q * d, sib.begin() + (q + 1) * d);
        }
        return out;
    }
    /* MerkleTree::leaves, packed row-major [n_leaves][leaf_len] (copied from the device on first use) */
    const std::vector<F>& leaves() const {
        if (!have_leaves_) {
            leaves_.assign(n_leaves() * leaf_len(), 0);
            ctx_->check(gl_tree_read(ctx_->raw(), h_, GL_PART_LEAVES, leaves_.data()));
            have_leaves_ = true;
        }
        return leaves_;
    }
    /* MerkleTree::digests in upstream's interleaved per-subtree layout, 2*(n_leaves - 2^cap_height) hashes */
    const std::vector<HashOut>& digests() const {
        if (!have_digests_) {
            digests_.assign(2 * (n_leaves() - (size_t(1) << cap_height())), HashOut{});
            if (!digests_.empty()) ctx_->check(gl_tree_read(ctx_->raw(), h_, GL_PART_DIGESTS, digests_[0].elements.data()));
            have_digests_ = true;
        }
        return digests_;
    }

private:
    void release() {
        if (h_ && ctx_ && ctx_->raw()) gl_tree_free(ctx_->raw(), h_);
        h_ = 0;
    }
    Context* ctx_ = nullptr;
    gl_handle h_ = 0;
    gl_tree_info_t info_{};
    mutable std::vector<F> leaves_;
    mutable std::vector<HashOut> digests_;
    mutable bool have_leaves_ = false, have_digests_ = false;
};

/* ------------------------------------------------------------------------------------------------ Challenger */
/* plonky2 iop/challenger.rs · Challenger<F, PoseidonHash>: duplex sponge in overwrite mode; the permutation runs on the
 * device (gl_poseidon_permute).  The three fields are public because fri_proof_of_work reads them, as upstream does. */
class Challenger {
public:
    std::array<F, SPONGE_WIDTH> sponge_state{};
    std::vector<F> input_buffer, output_buffer;

    explicit Challenger(Context* ctx = nullptr) : ctx_(&ctx_or_default(ctx)) {}

    void observe_element(F e) {
        output_buffer.clear();                       /* any buffered outputs are now invalid */
        input_buffer.push_back(e >= ORDER ? e - ORDER : e);
        if (input_buffer.size() == SPONGE_RATE) duplexing();
    }
    /* observe_element for every element; the duplexing of all full groups of 8 runs in ONE device call (gl_poseidon_absorb): the chain of
     * permutations is sequential anyway, so a Merkle cap costs one launch and one round trip instead of eight */
    void observe_elements(const F* es, size_t n) {
        if (n == 0) return;
        output_buffer.clear();
        std::vector<F> buf(input_buffer);
        for (size_t i = 0; i < n; i++) buf.push_back(es[i] >= ORDER ? es[i] - ORDER : es[i]);
        const size_t n_full = buf.size() / SPONGE_RATE;
        if (n_full) {
            ctx_->check(gl_poseidon_absorb(ctx_->raw(), sponge_state.data(), buf.data(), uint32_t(n_full)));
            output_buffer.assign(sponge_state.begin(), sponge_state.begin() + SPONGE_RATE);
        }
        input_buffer.assign(buf.begin() + n_full * SPONGE_RATE, buf.end());
        if (!input_buffer.empty()) output_buffer.clear();
    }
    void observe_elements(const std::vector<F>& es) { observe_elements(es.data(), es.size()); }
    void observe_hash(const HashOut& h) { observe_elements(h.elements.data(), 4); }
    void observe_cap(const MerkleCap& cap) { for (const auto& h : cap.hashes) observe_hash(h); }
    void observe_extension_element(const Ext& e) { observe_elements(e.data(), 2); }
    void observe_extension_elements(const std::vector<Ext>& es) { for (const auto& e : es) observe_extension_element(e); }
    /* every batch's values, in order (upstream: challenger.observe_openings(&openings.to_fri_openings())) */
    void observe_openings(const FriOpenings& openings) {
        for (const auto& b : openings.batches)
            if (!b.values.empty()) observe_elements(b.values[0].data(), 2 * b.values.size());
    }

    F get_challenge() {
        if (!input_buffer.empty() || output_buffer.empty()) duplexing();
        F v = output_buffer.back();
        output_buffer.pop_back();
        return v;
    }
    std::vector<F> get_n_challenges(size_t n) { std::vector<F> v(n); for (auto& x : v) x = get_challenge(); return v; }
    HashOut get_hash() { HashOut h; for (auto& x : h.elements) x = get_challenge(); return h; }
    Ext get_extension_challenge() { Ext e; e[0] = get_challenge(); e[1] = get_challenge(); return e; }
    std::vector<Ext> get_n_extension_challenges(size_t n) { std::vector<Ext> v(n); for (auto& x : v) x = get_extension_challenge(); return v; }

    Context& context() const { return *ctx_; }

private:
    void duplexing() {
        for (size_t i = 0; i < input_buffer.size(); i++) sponge_state[i] = input_buffer[i];
        input_buffer.clear();
        ctx_->poseidon_permute(sponge_state.data(), 1);
        output_buffer.assign(sponge_state.begin(), sponge_state.begin() + SPONGE_RATE);
    }
    Context* ctx_;
};

/* ------------------------------------------------------------------------------------------------ FRI structures */
/* plonky2 fri/reduction_strategies.rs · FriReductionStrategy (Fixed / ConstantArityBits; MinSize is a search over the latter's
 * parameter and is not used by standard_recursion_config) */
struct FriReductionStrategy {
    enum Kind { Fixed, ConstantArityBits } kind = ConstantArityBits;
    std::vector<size_t> fixed;                /* Fixed(arity_bits) */
    size_t arity_bits = 4, final_poly_bits = 5;   /* ConstantArityBits(4, 5): standard_recursion_config */
    std::vector<size_t> reduction_arity_bits(size_t degree_bits, size_t rate_bits, size_t cap_height, size_t /*num_queries*/) const {
        if (kind == Fixed) return fixed;
        std::vector<size_t> result;
        while (degree_bits > final_poly_bits && degree_bits + rate_bits - arity_bits >= cap_height) {
            result.push_back(arity_bits);
            if (degree_bits < arity_bits) throw Panic("assertion failed: degree_bits >= *arity_bits");
            degree_bits -= arity_bits;
        }
        return result;
    }
};
struct FriParams;
struct FriConfig {                            /* plonky2 fri/mod.rs; defaults = CircuitConfig::standard_recursion_config().fri_config */
    size_t rate_bits = 3, cap_height = 4;
    uint32_t proof_of_work_bits = 16;
    FriReductionStrategy reduction_strategy;
    size_t num_query_rounds = 28;
    inline FriParams fri_params(size_t degree_bits, bool hiding) const;
};
struct FriParams {
    FriConfig config;
    bool hiding = false;
    size_t degree_bits = 0;
    std::vector<size_t> reduction_arity_bits;
    size_t lde_bits() const { return degree_bits + config.rate_bits; }
    size_t lde_size() const { return size_t(1) << lde_bits(); }
    size_t total_arities() const { size_t t = 0; for (size_t a : reduction_arity_bits) t += a; return t; }
    size_t final_poly_bits() const { return degree_bits - total_arities(); }
    size_t final_poly_len() const { return size_t(1) << final_poly_bits(); }
};
/* FriConfig::fri_params(degree_bits, hiding) */
inline FriParams FriConfig::fri_params(size_t degree_bits, bool hiding) const {
    FriParams p;
    p.config = *this;
    p.hiding = hiding;
    p.degree_bits = degree_bits;
    p.reduction_arity_bits = reduction_strategy.reduction_arity_bits(degree_bits, rate_bits, cap_height, num_query_rounds);
    return p;
}
struct FriPolynomialInfo { size_t oracle_index, polynomial_index; };
struct FriBatchInfo { Ext point; std::vector<FriPolynomialInfo> polynomials; };
struct FriOracleInfo { size_t num_polys = 0; bool blinding = false; };
struct FriInstanceInfo { std::vector<FriOracleInfo> oracles; std::vector<FriBatchInfo> batches; };

struct FriInitialTreeProof { std::vector<std::pair<std::vector<F>, MerkleProof>> evals_proofs; };
struct FriQueryStep { std::vector<Ext> evals; MerkleProof merkle_proof; };
struct FriQueryRound { FriInitialTreeProof initial_trees_proof; std::vector<FriQueryStep> steps; };
struct FriProof {
    std::vector<MerkleCap> commit_phase_merkle_caps;
    std::vector<FriQueryRound> query_round_proofs;
    PolynomialCoeffsExt final_poly;
    F pow_witness = 0;
};

namespace detail {
/* owns a gl_fri state handle */
struct FriState {
    Context& ctx;
    gl_handle h = 0;
    explicit FriState(Context& c) : ctx(c) {}
    ~FriState() { if (h) gl_fri_end(ctx.raw(), h); }
    FriState(const FriState&) = delete;
    FriState& operator=(const FriState&) = delete;
};

/* the per-layer loop of fri_committed_trees on a device-resident FRI state */
inline std::pair<std::vector<MerkleTree>, PolynomialCoeffsExt> commit_phase(Context& ctx, gl_handle fri, Challenger& challenger,
                                                                            const FriParams& p) {
    std::vector<MerkleTree> trees;
    uint64_t cur = 0;
    ctx.check(gl_fri_read(ctx.raw(), fri, nullptr, nullptr, &cur));
    for (size_t arity_bits : p.reduction_arity_bits) {
        cur = arity_bits < 64 ? cur >> arity_bits : 0;   /* leaves of this layer: MerkleTree::new's assert, before the cap is sized */
        if (p.config.cap_height > 31 || (cur != 0 && (uint64_t(1) << p.config.cap_height) > cur))   /* cur == 0: the library reports the arity */
            throw Panic("cap_height=" + std::to_string(p.config.cap_height) + " should be at most log2(leaves.len())");
        MerkleCap cap;
        cap.hashes.resize(size_t(1) << p.config.cap_height);
        gl_handle th = 0;
        ctx.check(gl_fri_commit_layer(ctx.raw(), fri, uint32_t(arity_bits), nullptr, nullptr, cap.hashes[0].elements.data(), &th));
        trees.emplace_back(ctx, th, std::move(cap));
        challenger.observe_cap(trees.back().cap);
        Ext beta = challenger.get_extension_challenge();
        ctx.check(gl_fri_fold(ctx.raw(), fri, beta.data()));
    }
    uint64_t n = 0;
    ctx.check(gl_fri_final_poly(ctx.raw(), fri, nullptr, &n));
    PolynomialCoeffsExt fin;
    fin.coeffs.resize(n);
    if (n) ctx.check(gl_fri_final_poly(ctx.raw(), fri, fin.coeffs[0].data(), &n));
    challenger.observe_extension_elements(fin.coeffs);
    return {std::move(trees), std::move(fin)};
}
}  // namespace detail

/* plonky2 fri/prover.rs · fri_committed_trees(coeffs, values, challenger, fri_params): values = coeffs.coset_fft(7) in
 * natural order, exactly the two arguments upstream passes. */
inline std::pair<std::vector<MerkleTree>, PolynomialCoeffsExt> fri_committed_trees(const PolynomialCoeffsExt& coeffs,
                                                                                   const PolynomialValuesExt& values,
                                                                                   Challenger& challenger, const FriParams& fri_params,
                                                                                   Context* ctx = nullptr) {
    Context& c = ctx ? *ctx : challenger.context();
    if (coeffs.len() != values.len() || coeffs.len() == 0) throw Panic("fri_committed_trees: coeffs and values must have the same length");
    detail::FriState st(c);
    c.check(gl_fri_begin(c.raw(), coeffs.coeffs[0].data(), values.values[0].data(), coeffs.len(), uint32_t(fri_params.config.rate_bits),
                         uint32_t(fri_params.config.cap_height), &st.h));
    return detail::commit_phase(c, st.h, challenger, fri_params);
}

/* plonky2 fri/prover.rs · fri_proof_of_work(challenger, config): grind on the device for the SMALLEST witness (what the
 * serial `find` of the reference build returns), then advance the transcript as upstream: observe the witness, draw the
 * response, assert its leading zeros. */
inline F fri_proof_of_work(Challenger& challenger, const FriConfig& config, Context* ctx = nullptr) {
    Context& c = ctx ? *ctx : challenger.context();
    const uint32_t min_leading_zeros = config.proof_of_work_bits + (64 - 64);   /* + (64 - F::order().bits()) */
    uint64_t w = 0;
    c.check(gl_fri_pow(c.raw(), challenger.sponge_state.data(), challenger.input_buffer.empty() ? nullptr : challenger.input_buffer.data(),
                       uint32_t(challenger.input_buffer.size()), min_leading_zeros, &w));
    challenger.observe_element(w);
    const F resp = challenger.get_challenge();
    const uint32_t lz = resp ? uint32_t(__builtin_clzll(resp)) : 64;
    if (lz < min_leading_zeros) throw Panic("fri_proof_of_work: response does not have the required leading zeros");
    return w;
}

/* plonky2 fri/prover.rs · fri_prover_query_rounds / fri_prover_query_round.  Upstream draws x_index per round and reads
 * every tree row by row; no observation happens between the draws, so all indices are drawn first and every tree is
 * opened once for all rounds (gl_tree_open_batch). */
inline std::vector<FriQueryRound> fri_prover_query_rounds(const std::vector<const MerkleTree*>& initial_merkle_trees,
                                                          const std::vector<MerkleTree>& trees, Challenger& challenger, size_t n,
                                                          const FriParams& fri_params) {
    if (trees.size() != fri_params.reduction_arity_bits.size()) throw Panic("fri_prover_query_rounds: one tree per reduction layer expected");
    const size_t rounds = fri_params.config.num_query_rounds;
    std::vector<uint64_t> xs(rounds);
    for (auto& x : xs) x = challenger.get_challenge() % n;
    std::vector<FriQueryRound> out(rounds);
    for (const MerkleTree* t : initial_merkle_trees) {
        auto opened = t->open_batch(xs);
        for (size_t q = 0; q < rounds; q++) out[q].initial_trees_proof.evals_proofs.push_back(std::move(opened[q]));
    }
    std::vector<uint64_t> cur = xs, idx(rounds);
    for (size_t l = 0; l < trees.size(); l++) {
        const size_t arity_bits = fri_params.reduction_arity_bits[l], arity = size_t(1) << arity_bits;
        for (size_t q = 0; q < rounds; q++) idx[q] = cur[q] >> arity_bits;
        auto opened = trees[l].open_batch(idx);
        for (size_t q = 0; q < rounds; q++) {
            const std::vector<F>& leaf = opened[q].first;                  /* unflatten: arity extension elements */
            if (leaf.size() != 2 * arity) throw Panic("fri_prover_query_rounds: commit-phase leaf is not arity extension elements");
            FriQueryStep step;
            /* evals = unflatten(tree.get(x_index >> arity_bits)): ALL arity elements — validate_shape wants evals.len() == arity and
             * the verifier reads evals[x_index & (arity - 1)]; only FriProof::compress drops the queried element */
            step.evals.reserve(arity);
            for (size_t k = 0; k < arity; k++) step.evals.push_back(Ext{leaf[2 * k], leaf[2 * k + 1]});
            step.merkle_proof = std::move(opened[q].second);
            out[q].steps.push_back(std::move(step));
        }
        cur = idx;
    }
    return out;
}

/* plonky2 fri/prover.rs · fri_proof(initial_merkle_trees, lde_polynomial_coeffs, lde_polynomial_values, challenger, fri_params, timing) */
inline FriProof fri_proof(const std::vector<const MerkleTree*>& initial_merkle_trees, const PolynomialCoeffsExt& lde_polynomial_coeffs,
                          const PolynomialValuesExt& lde_polynomial_values, Challenger& challenger, const FriParams& fri_params,
                          TimingTree* = nullptr, Context* ctx = nullptr) {
    const size_t n = lde_polynomial_values.len();
    if (lde_polynomial_coeffs.len() != n) throw Panic("fri_proof: lde_polynomial_coeffs.len() != lde_polynomial_values.len()");
    auto committed = fri_committed_trees(lde_polynomial_coeffs, lde_polynomial_values, challenger, fri_params, ctx);
    FriProof proof;
    for (const auto& t : committed.first) proof.commit_phase_merkle_caps.push_back(t.cap);
    proof.final_poly = std::move(committed.second);
    proof.pow_witness = fri_proof_of_work(challenger, fri_params.config, ctx);
    proof.query_round_proofs = fri_prover_query_rounds(initial_merkle_trees, committed.first, challenger, n, fri_params);
    return proof;
}

/* ------------------------------------------------------------------------------------------------ PolynomialBatch */
/* plonky2 fri/oracle.rs · PolynomialBatch<GoldilocksField, PoseidonGoldilocksConfig, 2>
 * { polynomials, merkle_tree, degree_log, rate_bits, blinding } */
class PolynomialBatch {
public:
    MerkleTree merkle_tree;
    size_t degree_log = 0, rate_bits = 0;
    bool blinding = false;

    PolynomialBatch() = default;
    PolynomialBatch(PolynomialBatch&&) = default;
    PolynomialBatch& operator=(PolynomialBatch&&) = default;

    /* from_values(values, rate_bits, blinding, cap_height, timing, fft_root_table) */
    static PolynomialBatch from_values(const std::vector<PolynomialValues>& values, size_t rate_bits, bool blinding, size_t cap_height,
                                       TimingTree* = nullptr, const FftRootTable* = nullptr, Context* ctx = nullptr) {
        std::vector<const uint64_t*> cols;
        size_t n = values.empty() ? 0 : values[0].len();
        for (const auto& v : values) {
            if (v.len() != n) throw Panic("Polynomial degrees inconsistent");
            cols.push_back(v.values.data());
        }
        return commit(cols, n, rate_bits, blinding, cap_height, 0, ctx);
    }
    /* from_coeffs(polynomials, rate_bits, blinding, cap_height, timing, fft_root_table) */
    static PolynomialBatch from_coeffs(const std::vector<PolynomialCoeffs>& polynomials, size_t rate_bits, bool blinding, size_t cap_height,
                                       TimingTree* = nullptr, const FftRootTable* = nullptr, Context* ctx = nullptr) {
        std::vector<const uint64_t*> cols;
        size_t n = polynomials.empty() ? 0 : polynomials[0].len();
        for (const auto& v : polynomials) {
            if (v.len() != n) throw Panic("Polynomial degrees inconsistent");
            cols.push_back(v.coeffs.data());
        }
        return commit(cols, n, rate_bits, blinding, cap_height, 1, ctx);
    }

    size_t num_polys() const { return merkle_tree.leaf_len(); }

    /* PolynomialBatch::polynomials — canonical coefficients, one vector per column (copied from the device on first use) */
    const std::vector<PolynomialCoeffs>& polynomials() const {
        if (polys_.empty()) {
            const size_t n = size_t(1) << degree_log, c = num_polys();
            std::vector<F> flat(n * c);
            Context& ctx = merkle_tree.context();
            ctx.check(gl_tree_read(ctx.raw(), merkle_tree.handle(), GL_PART_COEFFS, flat.data()));
            polys_.resize(c);
            for (size_t j = 0; j < c; j++) polys_[j].coeffs.assign(flat.begin() + j * n, flat.begin() + (j + 1) * n);
        }
        return polys_;
    }

    /* get_lde_values(index, step): leaves[reverse_bits(index * step, degree_log + rate_bits)] */
    std::vector<F> get_lde_values(size_t index, size_t step) const {
        std::vector<F> row(num_polys());
        Context& ctx = merkle_tree.context();
        ctx.check(gl_tree_get_lde_values(ctx.raw(), merkle_tree.handle(), index, step, row.data()));
        return row;
    }

    /* prove_openings(instance, oracles, challenger, fri_params, timing): alpha <- challenger; per batch reduce_polys_base,
     * divide_by_linear, shift_poly; final_poly.lde(rate_bits).coset_fft(7); fri_proof.  The coefficient matrices of the oracles
     * and the LDE of the final polynomial never leave HBM. */
    static FriProof prove_openings(const FriInstanceInfo& instance, const std::vector<const PolynomialBatch*>& oracles, Challenger& challenger,
                                   const FriParams& fri_params, TimingTree* = nullptr, Context* ctx = nullptr) {
        if (oracles.empty()) throw Panic("prove_openings: no oracles");
        Context& c = ctx ? *ctx : challenger.context();
        if (fri_params.hiding) throw Panic("GPU path: zero_knowledge is off in plonky2.5 (src/p3/mod.rs:231)");
        const size_t degree_log = oracles[0]->degree_log;
        const Ext alpha = challenger.get_extension_challenge();
        struct Openings {
            Context& ctx; gl_handle h = 0;
            ~Openings() { if (h) gl_openings_end(ctx.raw(), h); }
        } op{c};
        c.check(gl_openings_begin(c.raw(), uint32_t(degree_log), &op.h));
        for (const FriBatchInfo& batch : instance.batches) {
            std::vector<gl_handle> hs;
            std::vector<uint32_t> cs;
            for (const FriPolynomialInfo& fpi : batch.polynomials) {
                if (fpi.oracle_index >= oracles.size()) throw Panic("prove_openings: oracle_index out of range");
                hs.push_back(oracles[fpi.oracle_index]->merkle_tree.handle());
                cs.push_back(uint32_t(fpi.polynomial_index));
            }
            c.check(gl_openings_add_batch(c.raw(), op.h, hs.empty() ? nullptr : hs.data(), cs.empty() ? nullptr : cs.data(), uint32_t(hs.size()),
                                          alpha.data(), batch.point.data(), nullptr));
        }
        detail::FriState st(c);
        c.check(gl_openings_lde(c.raw(), op.h, uint32_t(fri_params.config.rate_bits), uint32_t(fri_params.config.cap_height), &st.h));
        uint64_t lde_len = 0;
        c.check(gl_fri_read(c.raw(), st.h, nullptr, nullptr, &lde_len));
        auto committed = detail::commit_phase(c, st.h, challenger, fri_params);
        FriProof proof;
        for (const auto& t : committed.first) proof.commit_phase_merkle_caps.push_back(t.cap);
        proof.final_poly = std::move(committed.second);
        proof.pow_witness = fri_proof_of_work(challenger, fri_params.config, &c);
        std::vector<const MerkleTree*> initial;
        for (const PolynomialBatch* o : oracles) initial.push_back(&o->merkle_tree);
        proof.query_round_proofs = fri_prover_query_rounds(initial, committed.first, challenger, size_t(lde_len), fri_params);
        return proof;
    }

    /* from_values on several GPUs from this one process (gl_commit_multi): one Context per device.  The batch comes back as one
     * shard tree per context — leaf row i lives in shards[i / rows_per_shard] at local index i % rows_per_shard, and `prove` there is
     * MerkleTree::prove(i) — under the cap of the whole batch. */
    struct Sharded {
        MerkleCap cap;
        std::vector<MerkleTree> shards;
        size_t degree_log = 0, rate_bits = 0;
        size_t rows_per_shard() const { return shards.empty() ? 0 : shards[0].n_leaves(); }
        std::vector<F> get(size_t i) const { return shards[i / rows_per_shard()].get(i % rows_per_shard()); }
        MerkleProof prove(size_t i) const { return shards[i / rows_per_shard()].prove(i % rows_per_shard()); }
    };
    static Sharded from_values_multi(const std::vector<Context*>& ctxs, const std::vector<PolynomialValues>& values, size_t rate_bits, bool blinding,
                                     size_t cap_height) {
        if (blinding) throw Panic("blinding (zero_knowledge) is not on the GPU path: the reference runs with zk off (src/p3/mod.rs:231)");
        if (ctxs.empty() || !ctxs[0]) throw Panic("from_values_multi: no contexts");
        if (values.empty()) throw Panic("PolynomialBatch: empty polynomial batch");
        const size_t n = values[0].len();
        if (n == 0 || (n & (n - 1))) throw Panic("PolynomialBatch: polynomial length must be a power of two");
        {   /* upstream's assert, checked before the cap is sized by 2^cap_height */
            size_t lg = 0;
            while ((size_t(1) << lg) < n) lg++;
            if (cap_height > lg + rate_bits) throw Panic("cap_height=" + std::to_string(cap_height) + " should be at most log2(leaves.len())");
        }
        std::vector<const uint64_t*> cols;
        for (const auto& v : values) {
            if (v.len() != n) throw Panic("Polynomial degrees inconsistent");
            cols.push_back(v.values.data());
        }
        std::vector<gl_ctx*> raw;
        for (Context* c : ctxs) raw.push_back(c ? c->raw() : nullptr);
        size_t log_n = 0;
        while ((size_t(1) << log_n) < n) log_n++;
        Sharded out;
        out.cap.hashes.resize(size_t(1) << cap_height);
        out.degree_log = log_n;
        out.rate_bits = rate_bits;
        std::vector<gl_handle> hs(ctxs.size(), 0);
        ctxs[0]->check(gl_commit_multi(raw.data(), uint32_t(raw.size()), cols.data(), uint32_t(cols.size()), uint32_t(log_n), uint32_t(rate_bits),
                                       uint32_t(cap_height), 0, out.cap.hashes[0].elements.data(), hs.data()));
        const size_t per = out.cap.hashes.size() / ctxs.size();
        for (size_t g = 0; g < ctxs.size(); g++) {
            MerkleCap sub;
            sub.hashes.assign(out.cap.hashes.begin() + g * per, out.cap.hashes.begin() + (g + 1) * per);
            out.shards.emplace_back(*ctxs[g], hs[g], std::move(sub));
        }
        return out;
    }

private:
    static PolynomialBatch commit(const std::vector<const uint64_t*>& cols, size_t n, size_t rate_bits, bool blinding, size_t cap_height,
                                  int input_is_coeffs, Context* ctx) {
        if (blinding) throw Panic("blinding (zero_knowledge) is not on the GPU path: the reference runs with zk off (src/p3/mod.rs:231)");
        if (cols.empty()) throw Panic("PolynomialBatch: empty polynomial batch");
        if (n == 0 || (n & (n - 1))) throw Panic("PolynomialBatch: polynomial length must be a power of two");
        Context& c = ctx_or_default(ctx);
        size_t log_n = 0;
        while ((size_t(1) << log_n) < n) log_n++;
        /* upstream's assert, checked before the cap is sized by 2^cap_height */
        if (cap_height > log_n + rate_bits) throw Panic("cap_height=" + std::to_string(cap_height) + " should be at most log2(leaves.len())");
        MerkleCap cap;
        cap.hashes.resize(size_t(1) << cap_height);
        gl_handle h = 0;
        c.check(gl_commit(c.raw(), cols.data(), uint32_t(cols.size()), uint32_t(log_n), uint32_t(rate_bits), uint32_t(cap_height),
                          input_is_coeffs, nullptr, nullptr, nullptr, cap.hashes[0].elements.data(), &h));
        PolynomialBatch b;
        b.merkle_tree = MerkleTree(c, h, std::move(cap));
        b.degree_log = log_n;
        b.rate_bits = rate_bits;
        b.blinding = false;
        return b;
    }
    mutable std::vector<PolynomialCoeffs> polys_;

public:
    /* wrap a batch handle the library produced elsewhere (gl_quotient_commit) */
    static PolynomialBatch adopt(Context& c, gl_handle h, MerkleCap cap, size_t degree_log, size_t rate_bits) {
        PolynomialBatch b;
        b.merkle_tree = MerkleTree(c, h, std::move(cap));
        b.degree_log = degree_log;
        b.rate_bits = rate_bits;
        b.blinding = false;
        return b;
    }
};

/* ------------------------------------------------------------------------------------------------ OpeningSet */
/* OpeningSet::new's eval_commitment closure on the device (gl_batch_eval): every polynomial of `batch` at each of 1 or 2 extension
 * points; out[p][j] = polynomials[j].to_extension().eval(points[p]).  The coefficients stay in HBM. */
inline std::vector<std::vector<Ext>> eval_commitment(const PolynomialBatch& batch, const std::vector<Ext>& points) {
    Context& c = batch.merkle_tree.context();
    const size_t n = batch.num_polys();
    std::vector<Ext> flat(points.size() * n);
    c.check(gl_batch_eval(c.raw(), batch.merkle_tree.handle(), points.empty() ? nullptr : points[0].data(), uint32_t(points.size()),
                          flat.empty() ? nullptr : flat[0].data()));
    std::vector<std::vector<Ext>> out(points.size());
    for (size_t p = 0; p < points.size(); p++) out[p].assign(flat.begin() + p * n, flat.begin() + (p + 1) * n);
    return out;
}

/* plonky2 plonk/proof.rs · OpeningSet, without lookups (the reference's circuits use none) */
struct OpeningSet {
    std::vector<Ext> constants, plonk_sigmas, wires, plonk_zs, plonk_zs_next, partial_products, quotient_polys;

    /* OpeningSet::new(zeta, g, constants_sigmas, wires, zs_partial_products, quotient, common_data): four device calls, the Z commit at
     * zeta and g * zeta in one.  Commit #0 holds the constants first; commit #2 the Z polynomial of every challenge first
     * (gl_partial_products' order), then the partial products. */
    static OpeningSet new_(const Ext& zeta, const Ext& g, const PolynomialBatch& constants_sigmas, const PolynomialBatch& wires,
                           const PolynomialBatch& zs_partial_products, const PolynomialBatch& quotient, size_t num_constants,
                           size_t num_challenges) {
        if (num_constants > constants_sigmas.num_polys() || num_challenges > zs_partial_products.num_polys())
            throw Panic("OpeningSet::new: num_constants / num_challenges exceed the width of their commit");
        auto mul = [](uint64_t a, uint64_t b) { return uint64_t((unsigned __int128)(a % ORDER) * (b % ORDER) % ORDER); };
        auto add = [](uint64_t a, uint64_t b) { return uint64_t(((unsigned __int128)a + b) % ORDER); };
        const Ext gz = {add(mul(g[0], zeta[0]), mul(7, mul(g[1], zeta[1]))), add(mul(g[0], zeta[1]), mul(g[1], zeta[0]))};
        const auto cs = eval_commitment(constants_sigmas, {zeta})[0];
        const auto zs = eval_commitment(zs_partial_products, {zeta, gz});
        OpeningSet o;
        o.constants.assign(cs.begin(), cs.begin() + num_constants);
        o.plonk_sigmas.assign(cs.begin() + num_constants, cs.end());
        o.wires = eval_commitment(wires, {zeta})[0];
        o.plonk_zs.assign(zs[0].begin(), zs[0].begin() + num_challenges);
        o.plonk_zs_next.assign(zs[1].begin(), zs[1].begin() + num_challenges);
        o.partial_products.assign(zs[0].begin() + num_challenges, zs[0].end());
        o.quotient_polys = eval_commitment(quotient, {zeta})[0];
        return o;
    }

    /* the zeta batch (constants, sigmas, wires, zs, partial products, quotient) and the g * zeta batch (zs_next) */
    FriOpenings to_fri_openings() const {
        FriOpeningBatch at_zeta;
        for (const auto* v : {&constants, &plonk_sigmas, &wires, &plonk_zs, &partial_products, &quotient_polys})
            at_zeta.values.insert(at_zeta.values.end(), v->begin(), v->end());
        return FriOpenings{{std::move(at_zeta), FriOpeningBatch{plonk_zs_next}}};
    }
};

/* ------------------------------------------------------------------------------------------------ quotient / permutation / witness */
/* SURVEY §8(f) ranks 3-4.  Gate kinds are include/gl_commit.h's GL_GATE_* (the reference's own gates: Poseidon2Gate and the eight
 * u32 / b32 gates under /root/reference/src/common/u32/gates/; plonky2's Noop, Constant, PublicInput, Arithmetic, BaseSum, Poseidon,
 * Exponentiation and RandomAccess gates). */

/* Gate::eval_unfiltered_base_batch on host rows: rows = n x num_wires words -> n x num_constraints constraint values */
inline std::vector<F> evaluate_gate_constraints(int kind, uint32_t param, const std::vector<F>& rows, Context* ctx = nullptr) {
    Context& c = ctx_or_default(ctx);
    const int nw = gl_gate_num_wires(kind, param), nc = gl_gate_num_constraints(kind, param);
    if (nw <= 0 || nc <= 0) throw Panic("unknown gate kind / parameter");
    if (rows.size() % size_t(nw)) throw Panic("rows must be n * num_wires words");
    const size_t n = rows.size() / size_t(nw);
    std::vector<F> out(n * size_t(nc));
    c.check(gl_gate_eval_rows(c.raw(), kind, param, rows.data(), n, out.data()));
    return out;
}

/* plonky2 gates/selectors.rs · SelectorsInfo: gate i is filtered by selector column selector_indices[i], whose gate range is
 * groups[selector_indices[i]] = [first, second) */
struct SelectorsInfo {
    std::vector<size_t> selector_indices;
    std::vector<std::pair<size_t, size_t>> groups;
    size_t num_selectors() const { return groups.size(); }
};

/* the gate part of plonky2 plonk/prover.rs · compute_quotient_polys over the resident LDE rows of the wires commit, and its tail
 * (divide by Z_H on the coset, coset_ifft, chunks(degree), PolynomialBatch::from_coeffs) */
class QuotientAccumulator {
public:
    QuotientAccumulator(const PolynomialBatch& wires, size_t num_challenges, Context* ctx = nullptr);
    ~QuotientAccumulator() { if (h_) gl_quotient_end(ctx_->raw(), h_); }
    QuotientAccumulator(const QuotientAccumulator&) = delete;
    QuotientAccumulator& operator=(const QuotientAccumulator&) = delete;
    /* acc[k][row] += filter(row) * sum_i alphas[k]^(constraint_offset + i) * constraint_i(row) */
    void add_gate(int kind, uint32_t param, const std::vector<F>& alphas, size_t constraint_offset = 0, const PolynomialBatch* filter_batch = nullptr,
                  size_t filter_col = 0);
    /* plonk/vanishing_poly.rs · evaluate_gate_constraints_base_batch: gates[i] = (kind, param) of CommonCircuitData::gates; each gate's
     * constraints times compute_filter(i, group, s(x), num_selectors > 1), s its selector column of constants_sigmas (commit #0), gate
     * constants from the columns after the selectors; constraint c weighted by alphas[k]^(constraint_offset + c) */
    void add_gates(const std::vector<std::pair<int, uint32_t>>& gates, const SelectorsInfo& selectors_info, size_t num_lookup_selectors,
                   const PolynomialBatch& constants_sigmas, size_t num_constants, const HashOut& public_inputs_hash, const std::vector<F>& alphas,
                   size_t constraint_offset);
    /* the permutation-argument terms of eval_vanishing_poly_base_batch (vanishing_terms[0 .. n_ch * (1 + n_chunks))) */
    void add_permutation(const PolynomialBatch& sigmas, size_t sigma_col0, const PolynomialBatch& zs_partial_products, size_t n_routed, size_t degree,
                         const std::vector<F>& k_is, const std::vector<F>& betas, const std::vector<F>& gammas, const std::vector<F>& alphas) {
        if (k_is.size() != n_routed || betas.size() != n_challenges_ || gammas.size() != n_challenges_ || alphas.size() != n_challenges_)
            throw Panic("QuotientAccumulator::add_permutation: k_is per routed wire; betas / gammas / alphas per challenge");
        ctx_->check(gl_quotient_add_permutation(ctx_->raw(), h_, sigmas.merkle_tree.handle(), uint32_t(sigma_col0), zs_partial_products.merkle_tree.handle(),
                                                uint32_t(n_routed), uint32_t(degree), k_is.data(), betas.data(), gammas.data(), alphas.data()));
    }
    std::vector<F> values() const {                       /* [num_challenges][R], row order = the leaves' */
        std::vector<F> out(n_challenges_ * n_rows_);
        ctx_->check(gl_quotient_read(ctx_->raw(), h_, out.data()));
        return out;
    }
    PolynomialBatch commit(size_t cap_height);            /* quotient_polys_commitment */

private:
    Context* ctx_;
    gl_handle h_ = 0;
    size_t n_challenges_, n_rows_, degree_log_, rate_bits_;
};

/* plonk/prover.rs · all_wires_permutation_partial_products, columns in prove()'s order (Z of every challenge first) */
inline std::vector<PolynomialValues> partial_products_and_zs(const std::vector<PolynomialValues>& wires, const std::vector<PolynomialValues>& sigmas,
                                                             const std::vector<F>& k_is, const std::vector<F>& betas, const std::vector<F>& gammas,
                                                             size_t degree, Context* ctx = nullptr) {
    Context& c = ctx_or_default(ctx);
    if (wires.empty() || wires.size() != sigmas.size() || wires.size() != k_is.size()) throw Panic("partial_products: one sigma and one k_i per routed wire");
    if (betas.empty() || betas.size() != gammas.size()) throw Panic("partial_products: one (beta, gamma) per challenge");
    if (degree == 0) throw Panic("partial_products: degree must be positive");
    const size_t n = wires[0].len();
    if (n == 0 || (n & (n - 1))) throw Panic("partial_products: polynomial length must be a power of two");
    std::vector<const uint64_t*> wp, sp;
    for (size_t j = 0; j < wires.size(); j++) {
        if (wires[j].len() != n || sigmas[j].len() != n) throw Panic("Polynomial degrees inconsistent");
        wp.push_back(wires[j].values.data());
        sp.push_back(sigmas[j].values.data());
    }
    size_t log_n = 0;
    while ((size_t(1) << log_n) < n) log_n++;
    const size_t n_chunks = (wires.size() + degree - 1) / degree, n_out = betas.size() * n_chunks;
    std::vector<F> flat(n_out * n);
    c.check(gl_partial_products(c.raw(), wp.data(), sp.data(), uint32_t(wires.size()), uint32_t(log_n), k_is.data(), betas.data(), gammas.data(),
                                uint32_t(betas.size()), uint32_t(degree), flat.data()));
    std::vector<PolynomialValues> out(n_out);
    for (size_t j = 0; j < n_out; j++) out[j].values.assign(flat.begin() + j * n, flat.begin() + (j + 1) * n);
    return out;
}

/* /root/reference/src/common/poseidon2/poseidon2_gate.rs:447-523 · Poseidon2Generator::run_once for n rows: inputs n x 13 -> n x 135 */
inline std::vector<F> poseidon2_gate_witness(const std::vector<F>& inputs, Context* ctx = nullptr) {
    Context& c = ctx_or_default(ctx);
    if (inputs.size() % 13) throw Panic("poseidon2_gate_witness: inputs must be n * 13 words (12 state inputs + swap)");
    const size_t n = inputs.size() / 13;
    std::vector<F> out(n * 135);
    c.check(gl_poseidon2_gate_witness(c.raw(), inputs.data(), n, out.data()));
    return out;
}

/* plonky2 gates/poseidon.rs · PoseidonGenerator::run_once for n PoseidonGate rows: inputs n x 13 -> n x 135 */
inline std::vector<F> poseidon_gate_witness(const std::vector<F>& inputs, Context* ctx = nullptr) {
    Context& c = ctx_or_default(ctx);
    if (inputs.size() % 13) throw Panic("poseidon_gate_witness: inputs must be n * 13 words (12 state inputs + swap)");
    const size_t n = inputs.size() / 13;
    std::vector<F> out(n * 135);
    c.check(gl_poseidon_gate_witness(c.raw(), inputs.data(), n, out.data()));
    return out;
}

inline QuotientAccumulator::QuotientAccumulator(const PolynomialBatch& wires, size_t num_challenges, Context* ctx)
    : ctx_(&ctx_or_default(ctx)), n_challenges_(num_challenges), n_rows_(wires.merkle_tree.n_leaves()), degree_log_(wires.degree_log),
      rate_bits_(wires.rate_bits) {
    ctx_->check(gl_quotient_begin(ctx_->raw(), wires.merkle_tree.handle(), uint32_t(num_challenges), &h_));
}
inline void QuotientAccumulator::add_gate(int kind, uint32_t param, const std::vector<F>& alphas, size_t constraint_offset,
                                          const PolynomialBatch* filter_batch, size_t filter_col) {
    if (alphas.size() != n_challenges_) throw Panic("QuotientAccumulator::add_gate: one alpha per challenge expected");
    ctx_->check(gl_quotient_add_gate(ctx_->raw(), h_, kind, param, alphas.data(), uint32_t(constraint_offset),
                                     filter_batch ? filter_batch->merkle_tree.handle() : 0, uint32_t(filter_col)));
}
inline void QuotientAccumulator::add_gates(const std::vector<std::pair<int, uint32_t>>& gates, const SelectorsInfo& selectors_info,
                                           size_t num_lookup_selectors, const PolynomialBatch& constants_sigmas, size_t num_constants,
                                           const HashOut& public_inputs_hash, const std::vector<F>& alphas, size_t constraint_offset) {
    if (alphas.size() != n_challenges_) throw Panic("QuotientAccumulator::add_gates: one alpha per challenge expected");
    if (selectors_info.selector_indices.size() != gates.size()) throw Panic("QuotientAccumulator::add_gates: one selector index per gate expected");
    std::vector<int> kinds;
    std::vector<uint32_t> params, sel, groups;
    for (const auto& g : gates) { kinds.push_back(g.first); params.push_back(g.second); }
    for (size_t i : selectors_info.selector_indices) sel.push_back(uint32_t(i));
    for (const auto& r : selectors_info.groups) { groups.push_back(uint32_t(r.first)); groups.push_back(uint32_t(r.second)); }
    ctx_->check(gl_quotient_add_gates(ctx_->raw(), h_, kinds.data(), params.data(), uint32_t(kinds.size()), sel.data(), groups.data(),
                                      uint32_t(selectors_info.num_selectors()), uint32_t(num_lookup_selectors), constants_sigmas.merkle_tree.handle(),
                                      uint32_t(num_constants), public_inputs_hash.elements.data(), alphas.data(), uint32_t(constraint_offset)));
}
inline PolynomialBatch QuotientAccumulator::commit(size_t cap_height) {
    if (cap_height > degree_log_ + rate_bits_) throw Panic("cap_height=" + std::to_string(cap_height) + " should be at most log2(leaves.len())");
    MerkleCap cap;
    cap.hashes.resize(size_t(1) << cap_height);
    gl_handle h = 0;
    ctx_->check(gl_quotient_commit(ctx_->raw(), h_, uint32_t(cap_height), cap.hashes[0].elements.data(), &h));
    return PolynomialBatch::adopt(*ctx_, h, std::move(cap), degree_log_, rate_bits_);
}

}  // namespace plonky2
#endif /* GL_PLONKY2_HPP */
