#include "device_bridge.hpp"

#include <map>
#include <mutex>
#include <stdexcept>
#include <string>
#include <tuple>

namespace qkd_b200
{
    namespace
    {
        using matrix_key = std::tuple<const void *, const void *, size_t, size_t>;
        matrix_key key_of(const H_matrix &h) { return {h.bit_nodes, h.check_nodes, h.num_bit_nodes, h.num_check_nodes}; }

        struct registry
        {
            std::mutex mu;
            std::map<matrix_key, qlb_code *> codes;
            std::vector<qlb_ctx *> all_contexts;
            ~registry()
            {
                for (qlb_ctx *c : all_contexts)
                    qlb_ctx_destroy(c);
                for (auto &kv : codes)
                    qlb_code_destroy(kv.second);
            }
        };
        registry &reg()
        {
            static registry r;
            return r;
        }
        thread_local std::map<int, qlb_ctx *> tl_contexts;
    }

    void check(int status, const char *what)
    {
        if (status != QLB_OK)
            throw std::runtime_error(std::string(what) + ": " + qlb_last_error());
    }

    // prefix sums of the node weights; `contiguous`: every row starts where the previous one ends (a matrix loaded by
    // read_sparse_alist_matrix / read_dense_matrix: its rows are slices of one flat array, matrix_io.cpp)
    static bool offsets_of(int *const *rows, const int *weights, size_t count, std::vector<int32_t> &ptr)
    {
        ptr.assign(count + 1, 0);
        bool contiguous = true;
        for (size_t i = 0; i < count; ++i)
        {
            ptr[i + 1] = ptr[i] + weights[i];
            contiguous &= rows[i] == rows[0] + ptr[i];
        }
        return contiguous;
    }

    flat_matrix flatten(const H_matrix &h)
    {
        flat_matrix f;
        f.n = static_cast<int32_t>(h.num_bit_nodes);
        f.m = static_cast<int32_t>(h.num_check_nodes);
        if (!offsets_of(h.check_nodes, h.check_nodes_weight, h.num_check_nodes, f.row_ptr))
            for (size_t j = 0; j < h.num_check_nodes; ++j) // rows allocated one by one (the reference's own layout): gather them
                f.col_idx.insert(f.col_idx.end(), h.check_nodes[j], h.check_nodes[j] + h.check_nodes_weight[j]);
        if (!offsets_of(h.bit_nodes, h.bit_nodes_weight, h.num_bit_nodes, f.col_ptr))
            for (size_t i = 0; i < h.num_bit_nodes; ++i)
                f.row_idx.insert(f.row_idx.end(), h.bit_nodes[i], h.bit_nodes[i] + h.bit_nodes_weight[i]);
        return f;
    }

    qlb_code *code_for(const H_matrix &h)
    {
        std::lock_guard<std::mutex> lk(reg().mu);
        auto it = reg().codes.find(key_of(h));
        if (it != reg().codes.end())
            return it->second;
        const flat_matrix f = flatten(h);
        // loaded matrices are CSR / CSC already: their arrays go to the library as they are
        const int32_t *col_idx = f.col_idx.empty() && h.num_check_nodes ? h.check_nodes[0] : f.col_idx.data();
        const int32_t *row_idx = f.row_idx.empty() && h.num_bit_nodes ? h.bit_nodes[0] : f.row_idx.data();
        qlb_code *code = nullptr;
        check(qlb_code_create(f.n, f.m, f.row_ptr.data(), col_idx, f.col_ptr.data(), row_idx, &code), "qlb_code_create");
        reg().codes.emplace(key_of(h), code);
        return code;
    }

    void forget_matrix(const H_matrix &h)
    {
        std::lock_guard<std::mutex> lk(reg().mu);
        auto it = reg().codes.find(key_of(h));
        if (it != reg().codes.end())
        {
            qlb_code_destroy(it->second);
            reg().codes.erase(it);
        }
    }

    int usable_devices() { return qlb_device_count(); }

    qlb_ctx *context(int device)
    {
        auto it = tl_contexts.find(device);
        if (it != tl_contexts.end())
            return it->second;
        qlb_ctx *ctx = nullptr;
        check(qlb_ctx_create(device, &ctx), "qlb_ctx_create");
        tl_contexts[device] = ctx;
        std::lock_guard<std::mutex> lk(reg().mu);
        reg().all_contexts.push_back(ctx);
        return ctx;
    }

    void release_device_state()
    {
        std::lock_guard<std::mutex> lk(reg().mu);
        for (qlb_ctx *c : reg().all_contexts)
            qlb_ctx_destroy(c);
        reg().all_contexts.clear();
        tl_contexts.clear();
        for (auto &kv : reg().codes)
            qlb_code_destroy(kv.second);
        reg().codes.clear();
    }

    qlb_decode_params params_from_cfg(size_t max_iterations, double threshold)
    {
        qlb_decode_params p{};
        p.precision = CFG.DEVICE_PRECISION == 32 ? QLB_PRECISION_F32 : QLB_PRECISION_F64;
        p.max_iterations = static_cast<int32_t>(max_iterations);
        p.enable_threshold = CFG.ENABLE_SUM_PRODUCT_MSG_LLR_THRESHOLD ? 1 : 0; // read inside the reference's decoder (:246,313)
        p.threshold = threshold;
        p.flags = (p.precision == QLB_PRECISION_F32 && CFG.DEVICE_FP32_FAST) ? QLB_FLAG_F32_FAST_MATH : 0;
        if (p.precision == QLB_PRECISION_F64 && CFG.DEVICE_FP64_FUSED)
            p.flags |= QLB_FLAG_F64_FUSED_RATIO;
        return p;
    }
}
