// Glue between the reference-style host API (qkd_ldpc.hpp) and the C-ABI (include/qkd_ldpc_b200.h).
#pragma once
#include <cstdint>
#include <memory>
#include <vector>

#include "qkd_ldpc.hpp"
#include "qkd_ldpc_b200.h"

namespace qkd_b200
{
    // An H_matrix in the C-ABI's input form: the offsets always; the index arrays only when the matrix's rows were allocated one
    // by one (empty for a matrix from read_*_matrix, whose rows are slices of flat CSR / CSC arrays that are passed as they are).
    struct flat_matrix
    {
        int32_t n = 0, m = 0;
        std::vector<int32_t> row_ptr, col_idx, col_ptr, row_idx;
    };
    flat_matrix flatten(const H_matrix &matrix);

    // Throws std::runtime_error carrying qlb_last_error() when `status` is not QLB_OK.
    void check(int status, const char *what);

    // The device code handle for `matrix` (created on first use, cached on the identity and shape of its arrays).
    qlb_code *code_for(const H_matrix &matrix);
    void forget_matrix(const H_matrix &matrix);

    // One context per (calling thread, device); created on first use. Throws when no B200 is usable.
    qlb_ctx *context(int device = 0);
    int usable_devices();

    qlb_decode_params params_from_cfg(size_t max_iterations, double threshold);
}
