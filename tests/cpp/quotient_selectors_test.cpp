// QuotientAccumulator::add_gates of include/gl_plonky2.hpp on the real library (tests/test_quotient_selectors.py builds and runs it on a
// GPU).  A circuit of 2^4 rows with PublicInputGate, ConstantGate, ArithmeticGate, BaseSumGate<2> and NoopGate under two selector groups:
// the committed quotient must satisfy Z_H(zeta) * sum_c zeta^(cN) t_c(zeta) = sum_c alpha^c * eval_filtered_c(zeta), with the filters and
// the gate constraints evaluated here on the host from the committed polynomials at zeta — and must not once a wire is tampered.
// Prints "ALL OK" and exits 0 on success.
#include <cstdio>
#include <cstdlib>
#include <string>
#include <utility>
#include <vector>

#include "gl_plonky2.hpp"

using namespace plonky2;

namespace {
constexpr uint64_t P = ORDER, UNUSED_SELECTOR = 0xFFFFFFFFULL;
uint64_t mul(uint64_t a, uint64_t b) { return uint64_t((unsigned __int128)(a % P) * (b % P) % P); }
uint64_t add(uint64_t a, uint64_t b) { return uint64_t(((unsigned __int128)(a % P) + (b % P)) % P); }
uint64_t sub(uint64_t a, uint64_t b) { return add(a, P - b % P); }
uint64_t pw(uint64_t b, uint64_t e) { uint64_t r = 1; for (; e; e >>= 1, b = mul(b, b)) if (e & 1) r = mul(r, b); return r; }
uint64_t horner(const std::vector<F>& f, uint64_t z) {
    uint64_t acc = 0;
    for (size_t k = f.size(); k-- > 0;) acc = add(mul(acc, z), f[k]);
    return acc;
}
uint64_t splitmix(uint64_t& s) {
    uint64_t z = (s += 0x9E3779B97F4A7C15ULL);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return (z ^ (z >> 31)) % P;
}

int failures = 0;
void check(bool ok, const std::string& what) {
    std::printf("%s %s\n", ok ? "ok  " : "FAIL", what.c_str());
    if (!ok) failures++;
}

constexpr size_t LOG_N = 4, N = size_t(1) << LOG_N, RATE_BITS = 3, N_WIRES = 135, NUM_SELECTORS = 2, NUM_CONSTANTS = NUM_SELECTORS + 2;
constexpr uint32_t BASE_SUM_PARAM = 8 | 2 << 8;   // BaseSumGate<2>, 8 limbs
const std::vector<std::pair<int, uint32_t>> GATES = {{GL_GATE_PUBLIC_INPUT, 0}, {GL_GATE_CONSTANT, 2}, {GL_GATE_ARITHMETIC, 20},
                                                     {GL_GATE_BASE_SUM, BASE_SUM_PARAM}, {GL_GATE_NOOP, 0}};
const SelectorsInfo SELECTORS = {{0, 0, 1, 1, 1}, {{0, 2}, {2, 5}}};

// eval_unfiltered of the gates above at one point (w: wires, k: gate constants, pi: public-inputs hash)
std::vector<uint64_t> gate_constraints(size_t i, const std::vector<uint64_t>& w, const uint64_t* k, const HashOut& pi) {
    std::vector<uint64_t> c;
    switch (GATES[i].first) {
        case GL_GATE_PUBLIC_INPUT: for (int j = 0; j < 4; j++) c.push_back(sub(w[j], pi.elements[j])); break;
        case GL_GATE_CONSTANT: for (int j = 0; j < 2; j++) c.push_back(sub(k[j], w[j])); break;
        case GL_GATE_ARITHMETIC:
            for (int j = 0; j < 20; j++) c.push_back(sub(w[4 * j + 3], add(mul(mul(w[4 * j], w[4 * j + 1]), k[0]), mul(w[4 * j + 2], k[1]))));
            break;
        case GL_GATE_BASE_SUM: {
            uint64_t acc = 0;
            for (int j = 7; j >= 0; j--) acc = add(mul(acc, 2), w[1 + j]);
            c.push_back(sub(acc, w[0]));
            for (int j = 0; j < 8; j++) c.push_back(mul(w[1 + j], sub(w[1 + j], 1)));
            break;
        }
        default: break;
    }
    return c;
}

// sum over gates of compute_filter(i, group, s, num_selectors > 1) * constraints_i, by constraint index
std::vector<uint64_t> eval_filtered(const std::vector<uint64_t>& w, const std::vector<uint64_t>& consts, const HashOut& pi) {
    std::vector<uint64_t> res;
    for (size_t i = 0; i < GATES.size(); i++) {
        const size_t s_idx = SELECTORS.selector_indices[i];
        const uint64_t s = consts[s_idx];
        uint64_t f = sub(UNUSED_SELECTOR, s);
        for (size_t j = SELECTORS.groups[s_idx].first; j < SELECTORS.groups[s_idx].second; j++)
            if (j != i) f = mul(f, sub(j, s));
        const auto c = gate_constraints(i, w, consts.data() + NUM_SELECTORS, pi);
        if (c.size() > res.size()) res.resize(c.size(), 0);
        for (size_t j = 0; j < c.size(); j++) res[j] = add(res[j], mul(f, c[j]));
    }
    return res;
}

// commit the circuit, run add_gates, commit the quotient, check the identity at zeta
bool identity_holds(Context& ctx, const std::vector<PolynomialValues>& wire_cols, const std::vector<PolynomialValues>& const_cols, const HashOut& pi,
                    uint64_t alpha, uint64_t zeta) {
    auto consts = PolynomialBatch::from_values(const_cols, RATE_BITS, false, 1, nullptr, nullptr, &ctx);
    auto wires = PolynomialBatch::from_values(wire_cols, RATE_BITS, false, 1, nullptr, nullptr, &ctx);
    QuotientAccumulator q(wires, 1, &ctx);
    q.add_gates(GATES, SELECTORS, 0, consts, NUM_CONSTANTS, pi, {alpha}, 0);
    auto t = q.commit(1);
    std::vector<uint64_t> ew, ec;
    for (const auto& p : wires.polynomials()) ew.push_back(horner(p.coeffs, zeta));
    for (const auto& p : consts.polynomials()) ec.push_back(horner(p.coeffs, zeta));
    const auto terms = eval_filtered(ew, ec, pi);
    uint64_t want = 0, a = 1;
    for (uint64_t v : terms) { want = add(want, mul(v, a)); a = mul(a, alpha); }
    uint64_t t_zeta = 0;
    const uint64_t zn = pw(zeta, N);
    for (size_t c = t.num_polys(); c-- > 0;) t_zeta = add(mul(t_zeta, zn), horner(t.polynomials()[c].coeffs, zeta));
    return mul(sub(zn, 1), t_zeta) == want;
}
}  // namespace

int main() {
    try {
        Context ctx(0);
        uint64_t seed = 7;
        HashOut pi;
        for (auto& e : pi.elements) e = splitmix(seed);
        // rows: 0 PublicInput, 1-2 Constant, 3-7 Arithmetic, 8-10 BaseSum, the rest Noop
        std::vector<size_t> row_gate(N, 4);
        row_gate[0] = 0;
        for (size_t r = 1; r < 3; r++) row_gate[r] = 1;
        for (size_t r = 3; r < 8; r++) row_gate[r] = 2;
        for (size_t r = 8; r < 11; r++) row_gate[r] = 3;
        std::vector<PolynomialValues> wires(N_WIRES), consts(NUM_CONSTANTS);
        for (auto& c : wires) { c.values.resize(N); for (auto& x : c.values) x = splitmix(seed); }   // unused wires stay random
        for (auto& c : consts) c.values.assign(N, 0);
        for (size_t r = 0; r < N; r++) {
            const size_t gi = row_gate[r], s = SELECTORS.selector_indices[gi];
            for (size_t j = 0; j < NUM_SELECTORS; j++) consts[j].values[r] = j == s ? gi : UNUSED_SELECTOR;
            auto w = [&](size_t j) -> uint64_t& { return wires[j].values[r]; };
            uint64_t* k = nullptr;
            switch (GATES[gi].first) {
                case GL_GATE_PUBLIC_INPUT: for (int j = 0; j < 4; j++) w(j) = pi.elements[j]; break;
                case GL_GATE_CONSTANT:
                    for (int j = 0; j < 2; j++) { consts[NUM_SELECTORS + j].values[r] = splitmix(seed); w(j) = consts[NUM_SELECTORS + j].values[r]; }
                    break;
                case GL_GATE_ARITHMETIC:
                    for (int j = 0; j < 2; j++) consts[NUM_SELECTORS + j].values[r] = splitmix(seed);
                    k = &consts[NUM_SELECTORS].values[r];
                    for (int j = 0; j < 20; j++)
                        w(4 * j + 3) = add(mul(mul(w(4 * j), w(4 * j + 1)), *k), mul(w(4 * j + 2), consts[NUM_SELECTORS + 1].values[r]));
                    break;
                case GL_GATE_BASE_SUM: {
                    const uint64_t v = splitmix(seed) & 0xFF;
                    w(0) = v;
                    for (int j = 0; j < 8; j++) w(1 + j) = (v >> j) & 1;
                    break;
                }
                default: break;
            }
        }
        const uint64_t alpha = splitmix(seed), zeta = splitmix(seed);
        check(identity_holds(ctx, wires, consts, pi, alpha, zeta), "Z_H(zeta) t(zeta) == vanishing(zeta) for a valid circuit");
        auto bad = wires;
        bad[2].values[1] = add(bad[2].values[1], 1);                                   // row 1 is a ConstantGate: wire 2 is unused there
        check(identity_holds(ctx, bad, consts, pi, alpha, zeta), "an unused wire does not matter");
        bad[5].values[9] = add(bad[5].values[9], 1);                                   // a limb of a BaseSumGate row
        check(!identity_holds(ctx, bad, consts, pi, alpha, zeta), "a tampered wire breaks the identity");
        HashOut other = pi;
        other.elements[3] = add(other.elements[3], 1);
        check(!identity_holds(ctx, wires, consts, other, alpha, zeta), "a different public-inputs hash breaks the identity");
        bool refused = false;
        try {
            auto wb = PolynomialBatch::from_values(wires, RATE_BITS, false, 1, nullptr, nullptr, &ctx);
            auto cb = PolynomialBatch::from_values(consts, RATE_BITS, false, 1, nullptr, nullptr, &ctx);
            QuotientAccumulator q(wb, 1, &ctx);
            q.add_gates(GATES, SelectorsInfo{{0, 0, 1, 1, 2}, {{0, 2}, {2, 5}}}, 0, cb, NUM_CONSTANTS, pi, {alpha}, 0);
        } catch (const Panic& e) {
            refused = std::string(e.what()).find("selector index 2 >= num_selectors 2") != std::string::npos;
        }
        check(refused, "an out-of-range selector index panics with the library's message");
    } catch (const std::exception& e) {
        std::printf("FAIL exception: %s\n", e.what());
        return 1;
    }
    if (failures) return 1;
    std::printf("ALL OK\n");
    return 0;
}
