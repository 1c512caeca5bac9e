// The reference's per-frame hot-path functions as batch-of-one calls into libqkdldpc_b200.so.
//   calculate_syndrome_regular / _irregular   <- reference src/array_and_matrix_operations.cpp:463-486
//   sum_product_decoding_regular / _irregular <- reference src/qkd_ldpc_algorithm.cpp:3-173 / 175-345
//   QKD_LDPC_regular / _irregular             <- reference src/qkd_ldpc_algorithm.cpp:347-396 / 398-447
// The *_regular variants of the reference loop over max_*_weight instead of the per-node weights; on a matrix whose
// header weights are consistent the two are the same function, and an inconsistent "regular" matrix is rejected here
// rather than read out of bounds.
// With CFG.TRACE_QKD_LDPC / TRACE_SUM_PRODUCT / TRACE_SUM_PRODUCT_LLR set, the same functions print what the reference prints
// (src/qkd_ldpc_algorithm.cpp:214-327, 407-442): the per-iteration E / L / z / s / M come from the device through
// qlb_sum_product_trace (fp64, one frame), so the trace shows the GPU decoder's own intermediates.
#include <algorithm>
#include <cmath>
#include <stdexcept>
#include <vector>

#include "device_bridge.hpp"
#include "qkd_ldpc.hpp"
#include "trace_print.hpp"

namespace
{
    void require_consistent_regular(const H_matrix &h)
    {
        for (size_t i = 0; i < h.num_bit_nodes; ++i)
            if (static_cast<size_t>(h.bit_nodes_weight[i]) != h.max_bit_nodes_weight)
                throw std::runtime_error("regular decoding requested on a matrix whose bit weights differ from max_bit_nodes_weight");
        for (size_t j = 0; j < h.num_check_nodes; ++j)
            if (static_cast<size_t>(h.check_nodes_weight[j]) != h.max_check_nodes_weight)
                throw std::runtime_error("regular decoding requested on a matrix whose check weights differ from max_check_nodes_weight");
    }

    void syndrome(const int *bits, const H_matrix &h, int *out)
    {
        qkd_b200::check(qlb_syndrome_batch(qkd_b200::context(), qkd_b200::code_for(h), 1, bits, out), "qlb_syndrome_batch");
    }

    using qkd_b200::colour;
    using qkd_b200::print_coloured;

    double max_abs(const std::vector<const double *> &rows, const std::vector<int> &len) // get_max_llr_* (src/array_and_matrix_operations.cpp:50-85)
    {
        double best = 0;
        for (size_t i = 0; i < rows.size(); ++i)
            for (int k = 0; k < len[i]; ++k)
            {
                const double a = std::fabs(rows[i][k]);
                if (a > best)
                    best = a;
            }
        return best;
    }

    // The decode with the reference's console trace; E / L / z / s / M are the device decoder's values.
    SP_result decode_traced(const double *llr, const H_matrix &h, const int *syndrome_in, size_t max_it, double thr, int *bits_out)
    {
        qlb_decode_params p = qkd_b200::params_from_cfg(max_it, thr);
        p.precision = QLB_PRECISION_F64; // the trace exists for the reference's arithmetic only
        p.flags = 0;
        p.min_sum_scale = 0.f;
        const size_t n = h.num_bit_nodes, m = h.num_check_nodes;
        size_t edges = 0;
        for (size_t j = 0; j < m; ++j)
            edges += static_cast<size_t>(h.check_nodes_weight[j]);
        const bool full = CFG.TRACE_SUM_PRODUCT;
        std::vector<double> e(max_it * edges), mm(max_it * edges), tot(full ? max_it * n : 0);
        std::vector<int> z(full ? max_it * n : 0), s(full ? max_it * m : 0);
        uint32_t iterations = 0;
        uint8_t result = 0;
        qkd_b200::check(qlb_sum_product_trace(qkd_b200::context(), qkd_b200::code_for(h), &p, llr, syndrome_in, static_cast<int32_t>(max_it), e.data(),
                                              full ? tot.data() : nullptr, full ? z.data() : nullptr, full ? s.data() : nullptr, mm.data(), bits_out,
                                              &iterations, &result),
                        "qlb_sum_product_trace");
        const bool success = (result & QLB_RES_SYNDROMES_MATCH) != 0;
        std::vector<int> bit_w(h.bit_nodes_weight, h.bit_nodes_weight + n), check_w(h.check_nodes_weight, h.check_nodes_weight + m);
        std::vector<const double *> e_rows(n), m_rows(m);
        double max_llr = 0.;
        for (size_t t = 0; t < iterations; ++t)
        {
            size_t q = 0;
            for (size_t i = 0; i < n; q += static_cast<size_t>(bit_w[i]), ++i)
                e_rows[i] = &e[t * edges + q];
            q = 0;
            for (size_t j = 0; j < m; q += static_cast<size_t>(check_w[j]), ++j)
                m_rows[j] = &mm[t * edges + q];
            if (full)
            {
                print_coloured(colour::blue, "\n\nIteration: " + std::to_string(t + 1) + "\n");
                print_coloured(colour::blue, "\nE:\n");
                print_irregular_matrix(e_rows.data(), n, bit_w.data());
                print_coloured(colour::blue, "\nL:\n");
                print_array(&tot[t * n], n);
                print_coloured(colour::blue, "\n\nz:\n");
                print_array(&z[t * n], n);
                print_coloured(colour::blue, "\n\ns:\n");
                print_array(&s[t * m], m);
            }
            if (success && t + 1 == iterations)
                break; // the reference returns before "M" and before folding this iteration into MAX_LLR (:285-298)
            if (full)
            {
                print_coloured(colour::blue, "\n\nM:\n");
                print_irregular_matrix(m_rows.data(), m, check_w.data());
            }
            if (CFG.TRACE_SUM_PRODUCT_LLR)
                max_llr = std::max({max_llr, max_abs(e_rows, bit_w), max_abs(m_rows, check_w)});
        }
        if (CFG.TRACE_SUM_PRODUCT_LLR)
            print_coloured(colour::blue, "\n\nMAX_LLR = " + qkd_b200::format_shortest(max_llr) + "\n");
        std::fflush(stdout);
        return {iterations, success};
    }

    SP_result decode(const double *llr, const H_matrix &h, const int *syndrome_in, size_t max_it, double thr, int *bits_out)
    {
        if (CFG.TRACE_SUM_PRODUCT || CFG.TRACE_SUM_PRODUCT_LLR)
            return decode_traced(llr, h, syndrome_in, max_it, thr, bits_out);
        const qlb_decode_params p = qkd_b200::params_from_cfg(max_it, thr);
        uint32_t iterations = 0;
        uint8_t result = 0;
        qkd_b200::check(qlb_sum_product_batch(qkd_b200::context(), qkd_b200::code_for(h), &p, 1, llr, syndrome_in, bits_out, &iterations, &result),
                        "qlb_sum_product_batch");
        return {iterations, (result & QLB_RES_SYNDROMES_MATCH) != 0};
    }

    // QKD_LDPC_* step by step, as the reference runs it, when anything is to be printed (src/qkd_ldpc_algorithm.cpp:398-447)
    LDPC_result reconcile_traced(const int *alice, const int *bob, double qber, const H_matrix &h)
    {
        const size_t n = h.num_bit_nodes, m = h.num_check_nodes;
        const double log_p = log((1. - qber) / qber);
        std::vector<double> apriori_llr(n);
        for (size_t i = 0; i < n; ++i)
            apriori_llr[i] = bob[i] ? -log_p : log_p;
        if (CFG.TRACE_QKD_LDPC)
        {
            print_coloured(colour::blue, "\nr:\n");
            print_array(apriori_llr.data(), n);
        }
        std::vector<int> alice_syndrome(m), bob_solution(n);
        syndrome(alice, h, alice_syndrome.data());
        if (CFG.TRACE_QKD_LDPC)
        {
            print_coloured(colour::blue, "\n\nAlice syndrome:\n");
            print_array(alice_syndrome.data(), m);
        }
        LDPC_result r;
        r.sp_res = decode(apriori_llr.data(), h, alice_syndrome.data(), CFG.SUM_PRODUCT_MAX_ITERATIONS, CFG.SUM_PRODUCT_MSG_LLR_THRESHOLD, bob_solution.data());
        if (CFG.TRACE_QKD_LDPC)
        {
            print_coloured(colour::blue, "\nBob corrected bit array:\n");
            print_array(bob_solution.data(), n);
        }
        r.keys_match = arrays_equal(alice, bob_solution.data(), n);
        if (CFG.TRACE_QKD_LDPC)
        {
            print_coloured(colour::blue, "\n\nIterations performed: " + std::to_string(r.sp_res.iterations_num) + "\n");
            print_coloured(colour::blue, std::string("Syndromes are match: ") + (r.sp_res.syndromes_match ? "YES" : "NO") + "\n");
            print_coloured(colour::blue, std::string("Keys are match: ") + (r.keys_match ? "YES" : "NO") + "\n");
        }
        std::fflush(stdout);
        return r;
    }

    LDPC_result reconcile(const int *alice, const int *bob, double qber, const H_matrix &h)
    {
        if (CFG.TRACE_QKD_LDPC || CFG.TRACE_SUM_PRODUCT || CFG.TRACE_SUM_PRODUCT_LLR)
            return reconcile_traced(alice, bob, qber, h);
        const qlb_decode_params p = qkd_b200::params_from_cfg(CFG.SUM_PRODUCT_MAX_ITERATIONS, CFG.SUM_PRODUCT_MSG_LLR_THRESHOLD);
        uint32_t iterations = 0;
        uint8_t result = 0;
        qkd_b200::check(qlb_reconcile_batch(qkd_b200::context(), qkd_b200::code_for(h), &p, 1, alice, bob, &qber, &iterations, &result, nullptr, nullptr),
                        "qlb_reconcile_batch");
        LDPC_result r;
        r.sp_res = {iterations, (result & QLB_RES_SYNDROMES_MATCH) != 0};
        r.keys_match = (result & QLB_RES_KEYS_MATCH) != 0;
        return r;
    }
}

void calculate_syndrome_regular(const int *const bit_array, const H_matrix &matrix, int *const syndrome_out)
{
    require_consistent_regular(matrix);
    syndrome(bit_array, matrix, syndrome_out);
}

void calculate_syndrome_irregular(const int *const bit_array, const H_matrix &matrix, int *const syndrome_out)
{
    syndrome(bit_array, matrix, syndrome_out);
}

SP_result sum_product_decoding_regular(const double *const bit_array_llr, const H_matrix &matrix, const int *const syndrome,
                                       const size_t &max_num_iterations, const double &msg_threshold, int *const bit_array_out)
{
    require_consistent_regular(matrix);
    return decode(bit_array_llr, matrix, syndrome, max_num_iterations, msg_threshold, bit_array_out);
}

SP_result sum_product_decoding_irregular(const double *const bit_array_llr, const H_matrix &matrix, const int *const syndrome,
                                         const size_t &max_num_iterations, const double &msg_threshold, int *const bit_array_out)
{
    return decode(bit_array_llr, matrix, syndrome, max_num_iterations, msg_threshold, bit_array_out);
}

LDPC_result QKD_LDPC_regular(const int *const alice_bit_array, const int *const bob_bit_array, const double &QBER, const H_matrix &matrix)
{
    require_consistent_regular(matrix);
    return reconcile(alice_bit_array, bob_bit_array, QBER, matrix);
}

LDPC_result QKD_LDPC_irregular(const int *const alice_bit_array, const int *const bob_bit_array, const double &QBER, const H_matrix &matrix)
{
    return reconcile(alice_bit_array, bob_bit_array, QBER, matrix);
}
