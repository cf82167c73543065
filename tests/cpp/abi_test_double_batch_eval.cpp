// TEST DOUBLE of gl_batch_eval (include/gl_commit.h) — test infrastructure, linked next to tests/cpp/abi_test_double.cpp so the CPU
// suite runs the OpeningSet host logic of include/gl_plonky2.hpp without a device.  Built only from the double's own entry points:
// gl_tree_info for the shape, gl_tree_read(GL_PART_COEFFS) for the coefficients (which also refuses a tree without coefficients with
// "tree has no coefficients" and sets the context's message), and the host Horner of tests/cpp/eval_ext_oracle.c.
#include <vector>

#include "gl_commit.h"

extern "C" {
void glo_eval_ext(const uint64_t* polys, uint32_t n_polys, uint64_t n, const uint64_t point[2], uint64_t* out);

int gl_batch_eval(gl_ctx* c, gl_handle h, const uint64_t* points, uint32_t n_points, uint64_t* out) {
    gl_tree_info_t info{};
    if (int rc = gl_tree_info(c, h, &info)) return rc;
    std::vector<uint64_t> coeffs((size_t(info.leaf_len) << info.degree_log) + 1);
    if (!info.has_coeffs) return gl_tree_read(c, h, GL_PART_COEFFS, coeffs.data());
    if (!points || !out || n_points == 0) return GL_ERR_INVALID;
    if (n_points > 2) return GL_ERR_UNSUPPORTED;
    if (int rc = gl_tree_read(c, h, GL_PART_COEFFS, coeffs.data())) return rc;
    for (uint32_t p = 0; p < n_points; p++)
        glo_eval_ext(coeffs.data(), info.leaf_len, uint64_t(1) << info.degree_log, points + 2 * p, out + 2 * uint64_t(p) * info.leaf_len);
    return GL_OK;
}
}  // extern "C"
