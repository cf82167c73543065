// plonky2's PoseidonGate, ExponentiationGate and RandomAccessGate through the C++ mirror (include/gl_plonky2.hpp) on the GPU,
// self-checking identities only (the word-for-word comparison with the oracle lives in tests/test_plonky2_std_gates.py):
//   * rows filled by poseidon_gate_witness satisfy every PoseidonGate constraint, and their outputs are the leaf hash's permutation
//     (gl_poseidon_permute) of the swapped inputs; a tampered wire breaks a constraint;
//   * a wires batch made of such a row (constant columns => every LDE row equals the row) accumulates a zero quotient;
//   * square-and-multiply rows satisfy ExponentiationGate, and a RandomAccessGate row without extra constants satisfies its gate;
//   * the shape queries agree with the header's formulas, and a RandomAccessGate with extra constants is refused by the entry points
//     without gate constants.
// Build: g++ -std=c++17 -O2 -I include tests/cpp/std_gates_test.cpp -o std_gates_test -L plonky2.5_b200 -lgl_commit
#include <cstdio>
#include <cstdlib>

#include "gl_plonky2.hpp"

using namespace plonky2;

static int failures = 0;
#define CHECK(cond, msg) do { if (!(cond)) { std::printf("FAIL: %s\n", msg); failures++; } } while (0)

static const uint64_t P = 0xFFFFFFFF00000001ULL;
static uint64_t mulp(uint64_t a, uint64_t b) { return uint64_t((unsigned __int128)a * b % P); }
static bool all_zero(const std::vector<F>& v) {
    for (F x : v)
        if (x != 0) return false;
    return true;
}

int main() {
    try {
        Context ctx(0);
        // (1) PoseidonGate witness rows
        std::vector<F> in;
        uint64_t z = 777;
        const int n = 8;
        for (int r = 0; r < n; r++) {
            for (int i = 0; i < 12; i++) { z = z * 6364136223846793005ULL + 1442695040888963407ULL; in.push_back(z % P); }
            in.push_back(uint64_t(r & 1));
        }
        std::vector<F> rows = poseidon_gate_witness(in, &ctx);
        CHECK(rows.size() == size_t(n) * 135, "witness size");
        std::vector<F> cons = evaluate_gate_constraints(GL_GATE_POSEIDON, 0, rows, &ctx);
        CHECK(cons.size() == size_t(n) * 123 && all_zero(cons), "generated rows satisfy all 123 PoseidonGate constraints");
        std::vector<F> states;
        for (int r = 0; r < n; r++)
            for (int i = 0; i < 12; i++) states.push_back(in[13 * r + ((r & 1) && i < 8 ? (i + 4) % 8 : i)]);
        ctx.check(gl_poseidon_permute(ctx.raw(), states.data(), n));
        bool same = true;
        for (int r = 0; r < n; r++)
            for (int i = 0; i < 12; i++) same = same && rows[135 * r + 12 + i] == states[12 * r + i];
        CHECK(same, "outputs equal gl_poseidon_permute of the swapped inputs");
        rows[135 + 70] ^= 1;   // a partial-round S-box input of row 1
        CHECK(!all_zero(evaluate_gate_constraints(GL_GATE_POSEIDON, 0, rows, &ctx)), "a tampered S-box wire breaks a constraint");
        rows[135 + 70] ^= 1;
        // (2) constant columns made of row 0: zero quotient
        const size_t N = 16;
        std::vector<PolynomialValues> wires(135);
        for (size_t j = 0; j < 135; j++) wires[j].values.assign(N, rows[j]);
        PolynomialBatch batch = PolynomialBatch::from_values(wires, 3, false, 2, nullptr, nullptr, &ctx);
        QuotientAccumulator q(batch, 2, &ctx);
        q.add_gate(GL_GATE_POSEIDON, 0, {7, 11});
        CHECK(all_zero(q.values()), "valid PoseidonGate rows accumulate a zero quotient");
        // (3) ExponentiationGate(n) rows: base^power by square-and-multiply, bits big-endian
        for (uint32_t nb : {1u, 17u, 66u}) {
            const uint64_t base = 0x123456789ULL + nb, power = nb == 66 ? 0xF0F0F0F0F0F0F0F1ULL : ((1ULL << nb) - 1) ^ 2;
            std::vector<F> w(2 + 2 * nb, 0);
            w[0] = base;
            uint64_t cur = 1;
            for (uint32_t i = 0; i < nb; i++) {
                const uint64_t bit = i < 64 ? (power >> i) & 1 : 0;
                w[1 + i] = bit;
            }
            for (uint32_t i = 0; i < nb; i++) {
                if (w[1 + nb - 1 - i]) cur = mulp(cur, base);
                w[2 + nb + i] = cur;
                cur = mulp(cur, cur);
            }
            w[1 + nb] = w[1 + 2 * nb];
            CHECK(gl_gate_num_wires(GL_GATE_EXPONENTIATION, nb) == int(2 + 2 * nb) && gl_gate_num_constraints(GL_GATE_EXPONENTIATION, nb) == int(nb + 1),
                  "ExponentiationGate shape");
            CHECK(all_zero(evaluate_gate_constraints(GL_GATE_EXPONENTIATION, nb, w, &ctx)), "ExponentiationGate witness satisfies the gate");
            w[1] ^= 1;
            CHECK(!all_zero(evaluate_gate_constraints(GL_GATE_EXPONENTIATION, nb, w, &ctx)), "a flipped power bit breaks ExponentiationGate");
        }
        // (4) RandomAccessGate, bits 3, 2 copies, no extra constants
        const uint32_t bits = 3, copies = 2, v = 1u << bits, param = bits | copies << 8;
        const uint32_t nw = (2 + v + bits) * copies;
        CHECK(gl_gate_num_wires(GL_GATE_RANDOM_ACCESS, param) == int(nw) && gl_gate_num_constraints(GL_GATE_RANDOM_ACCESS, param) == int((bits + 2) * copies) &&
              gl_gate_num_constants(GL_GATE_RANDOM_ACCESS, param) == 0, "RandomAccessGate shape");
        std::vector<F> w(nw, 0);
        for (uint32_t c = 0; c < copies; c++) {
            const uint32_t idx = 5 - 3 * c;
            w[(2 + v) * c] = idx;
            for (uint32_t i = 0; i < v; i++) w[(2 + v) * c + 2 + i] = 1000 * (c + 1) + i * i;
            w[(2 + v) * c + 1] = w[(2 + v) * c + 2 + idx];
            for (uint32_t i = 0; i < bits; i++) w[(2 + v) * copies + c * bits + i] = (idx >> i) & 1;
        }
        CHECK(all_zero(evaluate_gate_constraints(GL_GATE_RANDOM_ACCESS, param, w, &ctx)), "RandomAccessGate witness satisfies the gate");
        w[1] += 1;
        CHECK(!all_zero(evaluate_gate_constraints(GL_GATE_RANDOM_ACCESS, param, w, &ctx)), "a wrong claimed element breaks RandomAccessGate");
        // (5) a RandomAccessGate with extra constants needs the entry points with gate constants
        bool refused = false;
        try {
            q.add_gate(GL_GATE_RANDOM_ACCESS, 4 | 4 << 8 | 2 << 16, {7, 11});
        } catch (const std::exception& e) {
            refused = std::string(e.what()).find("gl_quotient_add_gates") != std::string::npos;
        }
        CHECK(refused, "RandomAccessGate with extra constants refused by add_gate");
        CHECK(gl_gate_num_wires(14, 0) == -1 && gl_gate_num_wires(GL_GATE_POSEIDON, 1) == -1 && gl_gate_num_wires(GL_GATE_EXPONENTIATION, 67) == -1,
              "refused kinds / params");
    } catch (const std::exception& e) {
        std::printf("FAIL: exception: %s\n", e.what());
        failures++;
    }
    std::printf(failures ? "FAILED (%d)\n" : "ALL OK\n", failures);
    return failures ? 1 : 0;
}
