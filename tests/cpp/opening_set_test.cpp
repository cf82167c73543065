// OpeningSet::new / to_fri_openings / Challenger::observe_openings of include/gl_plonky2.hpp.  Linked against the ABI test double on the
// CPU and against libgl_commit on a GPU (tests/test_opening_set.py).  Expected values come from a host Horner evaluation in this file,
// so the check does not depend on the library under test.  Prints "ALL OK" and exits 0 on success.
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

#include "gl_plonky2.hpp"

using namespace plonky2;

namespace {
constexpr uint64_t P = ORDER;
uint64_t mul(uint64_t a, uint64_t b) { return uint64_t((unsigned __int128)(a % P) * (b % P) % P); }
uint64_t add(uint64_t a, uint64_t b) { return uint64_t(((unsigned __int128)(a % P) + (b % P)) % P); }
Ext ext_mul(const Ext& a, const Ext& b) { return {add(mul(a[0], b[0]), mul(7, mul(a[1], b[1]))), add(mul(a[0], b[1]), mul(a[1], b[0]))}; }
Ext horner(const std::vector<F>& f, const Ext& z) {
    Ext acc = {0, 0};
    for (size_t k = f.size(); k-- > 0;) { acc = ext_mul(acc, z); acc[0] = add(acc[0], f[k]); }
    return acc;
}
uint64_t splitmix(uint64_t& s) {
    uint64_t z = (s += 0x9E3779B97F4A7C15ULL);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return z ^ (z >> 31);   // raw 64-bit words: non-canonical inputs on purpose
}

int failures = 0;
void check(bool ok, const std::string& what) {
    std::printf("%s %s\n", ok ? "ok  " : "FAIL", what.c_str());
    if (!ok) failures++;
}

template <class T>
std::vector<T> slice(const std::vector<T>& v, size_t a, size_t b) { return std::vector<T>(v.begin() + a, v.begin() + b); }

std::vector<Ext> expected(const PolynomialBatch& b, size_t c0, size_t c1, const Ext& z) {
    std::vector<Ext> out;
    for (size_t j = c0; j < c1; j++) out.push_back(horner(b.polynomials()[j].coeffs, z));
    return out;
}
}  // namespace

int main() {
    try {
        Context ctx(0);
        const size_t log_n = 5, n = size_t(1) << log_n, rate_bits = 1, cap_height = 1;
        const size_t widths[4] = {5, 7, 6, 4}, num_constants = 2, num_challenges = 2;
        uint64_t seed = 42;
        std::vector<PolynomialBatch> batches;
        for (int k = 0; k < 4; k++) {
            if (k < 3) {
                std::vector<PolynomialValues> v(widths[k]);
                for (auto& c : v) { c.values.resize(n); for (auto& x : c.values) x = splitmix(seed); }
                batches.push_back(PolynomialBatch::from_values(v, rate_bits, false, cap_height, nullptr, nullptr, &ctx));
            } else {
                std::vector<PolynomialCoeffs> v(widths[k]);
                for (auto& c : v) { c.coeffs.resize(n); for (auto& x : c.coeffs) x = splitmix(seed); }
                batches.push_back(PolynomialBatch::from_coeffs(v, rate_bits, false, cap_height, nullptr, nullptr, &ctx));
            }
        }
        const Ext zeta = {splitmix(seed), splitmix(seed)};
        uint64_t g = 1753635133440165772ULL;   // 2^32nd root of unity -> generator of the size-n subgroup
        for (size_t i = log_n; i < 32; i++) g = mul(g, g);
        const Ext gz = ext_mul({g, 0}, zeta);

        const OpeningSet os = OpeningSet::new_(zeta, {g, 0}, batches[0], batches[1], batches[2], batches[3], num_constants, num_challenges);
        check(os.constants == expected(batches[0], 0, num_constants, zeta), "constants = commit #0 columns [0, num_constants) at zeta");
        check(os.plonk_sigmas == expected(batches[0], num_constants, widths[0], zeta), "plonk_sigmas = the rest of commit #0 at zeta");
        check(os.wires == expected(batches[1], 0, widths[1], zeta), "wires at zeta");
        check(os.plonk_zs == expected(batches[2], 0, num_challenges, zeta), "plonk_zs = commit #2 columns [0, num_challenges) at zeta");
        check(os.plonk_zs_next == expected(batches[2], 0, num_challenges, gz), "plonk_zs_next = the same columns at g * zeta");
        check(os.partial_products == expected(batches[2], num_challenges, widths[2], zeta), "partial_products = the rest of commit #2 at zeta");
        check(os.quotient_polys == expected(batches[3], 0, widths[3], zeta), "quotient_polys at zeta");

        const FriOpenings fo = os.to_fri_openings();
        std::vector<Ext> want0;
        for (int k = 0; k < 4; k++) {
            auto e = expected(batches[k], 0, widths[k], zeta);
            want0.insert(want0.end(), e.begin(), e.end());
        }
        check(fo.batches.size() == 2, "two FRI opening batches");
        check(fo.batches[0].values == want0, "zeta batch = constants | sigmas | wires | zs | partial products | quotient (commit order)");
        check(fo.batches[1].values == os.plonk_zs_next, "g * zeta batch = plonk_zs_next");

        // transcript: observe_openings == every word of batch 0 then batch 1, one element at a time
        Challenger a(&ctx), b(&ctx), swapped(&ctx);
        a.observe_openings(fo);
        for (const auto& batch : fo.batches)
            for (const Ext& e : batch.values) { b.observe_element(e[0]); b.observe_element(e[1]); }
        swapped.observe_openings(FriOpenings{{fo.batches[1], fo.batches[0]}});
        const Ext ca = a.get_extension_challenge(), cb = b.get_extension_challenge(), cs = swapped.get_extension_challenge();
        check(ca == cb, "observe_openings observes the batches in order, element by element");
        check(ca != cs, "the batch order changes the transcript");

        // a tree without coefficients is refused with upstream's wording; more than two points are unsupported
        std::vector<F> leaves(16 * 3);
        for (auto& x : leaves) x = splitmix(seed);
        MerkleCap cap;
        cap.hashes.resize(1);
        gl_handle h = 0;
        ctx.check(gl_merkle_new(ctx.raw(), leaves.data(), 16, 3, 0, nullptr, cap.hashes[0].elements.data(), &h));
        const PolynomialBatch bare = PolynomialBatch::adopt(ctx, h, cap, 0, 0);
        bool refused = false;
        try {
            OpeningSet::new_(zeta, {g, 0}, batches[0], bare, batches[2], batches[3], num_constants, num_challenges);
        } catch (const Panic& p) {
            refused = std::string(p.what()).find("tree has no coefficients") != std::string::npos;
        }
        check(refused, "OpeningSet::new over a MerkleTree::new tree panics: tree has no coefficients");
        int code = 0;
        try { eval_commitment(batches[1], {zeta, gz, zeta}); } catch (const GlError& e) { code = e.code; }
        check(code == GL_ERR_UNSUPPORTED, "three points are GL_ERR_UNSUPPORTED");
        const auto two = eval_commitment(batches[1], {zeta, gz});
        check(two[0] == eval_commitment(batches[1], {zeta})[0] && two[1] == eval_commitment(batches[1], {gz})[0],
              "two points in one call == two one-point calls");
    } catch (const std::exception& e) {
        std::printf("FAIL exception: %s\n", e.what());
        return 1;
    }
    if (failures) return 1;
    std::printf("ALL OK\n");
    return 0;
}
