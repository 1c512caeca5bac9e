// config.json -> CFG. Same keys, validation and messages as the reference (src/config.cpp:4-115); the optional
// device_* keys default so that an unmodified reference config runs (fp64, all GPUs).
#include <algorithm>
#include <ctime>
#include <fstream>
#include <iostream>
#include <sstream>
#include <stdexcept>

#include "mini_json.hpp"
#include "qkd_ldpc.hpp"

config_data get_config_data(fs::path config_path)
{
    if (!fs::exists(config_path))
        throw std::runtime_error("Configuration file not found: " + config_path.string());
    std::ifstream in(config_path);
    if (!in.is_open())
        throw std::runtime_error("Failed to open configuration file: " + config_path.string());
    std::stringstream buf;
    buf << in.rdbuf();
    const mini_json::value root = mini_json::parse(buf.str());
    if (root.kind != mini_json::value::object_k || root.members.empty())
        throw std::runtime_error("Configuration file is empty: " + config_path.string());

    try
    {
        config_data cfg{};
        cfg.THREADS_NUMBER = root.at("threads_number").as_size();
        if (cfg.THREADS_NUMBER < 1)
            throw std::runtime_error("Number of threads must be >= 1!");
        cfg.TRIALS_NUMBER = root.at("trials_number").as_size();
        if (cfg.TRIALS_NUMBER < 1)
            throw std::runtime_error("Number of trials must be >= 1!");
        cfg.SIMULATION_SEED = root.at("use_config_simulation_seed").as_bool() ? root.at("simulation_seed").as_size()
                                                                              : static_cast<size_t>(std::time(nullptr));
        cfg.INTERACTIVE_MODE = root.at("interactive_mode").as_bool();
        cfg.SUM_PRODUCT_MAX_ITERATIONS = root.at("sum_product_max_iterations").as_size();
        if (cfg.SUM_PRODUCT_MAX_ITERATIONS < 1)
            throw std::runtime_error("Minimum number of sum-product iterations must be >= 1!");
        cfg.USE_DENSE_MATRICES = root.at("use_dense_matrices").as_bool();
        cfg.TRACE_QKD_LDPC = root.at("trace_qkd_ldpc").as_bool();
        cfg.TRACE_SUM_PRODUCT = root.at("trace_sum_product").as_bool();
        cfg.TRACE_SUM_PRODUCT_LLR = root.at("trace_sum_product_llr").as_bool();
        cfg.ENABLE_SUM_PRODUCT_MSG_LLR_THRESHOLD = root.at("enable_sum_product_msg_llr_threshold").as_bool();
        if (cfg.ENABLE_SUM_PRODUCT_MSG_LLR_THRESHOLD)
        {
            cfg.SUM_PRODUCT_MSG_LLR_THRESHOLD = root.at("sum_product_msg_llr_threshold").as_double();
            if (cfg.SUM_PRODUCT_MSG_LLR_THRESHOLD <= 0.)
                throw std::runtime_error("Sum-product message LLR threshold must be > 0!");
        }

        for (const auto &p : root.at("code_rate_QBER_parameters").items)
            cfg.R_QBER_PARAMETERS.push_back({p.at("code_rate").as_double(), p.at("QBER_begin").as_double(), p.at("QBER_end").as_double(),
                                             p.at("QBER_step").as_double()});
        if (cfg.R_QBER_PARAMETERS.empty())
            throw std::runtime_error("Array with code rate and QBER parameters is empty!");
        for (const auto &p : cfg.R_QBER_PARAMETERS)
        {
            if (p.code_rate <= 0. || p.code_rate >= 1.)
                throw std::runtime_error("Code rate(R) must be: 0 < R < 1!");
            if (p.QBER_begin <= 0. || p.QBER_begin >= 1. || p.QBER_end <= 0. || p.QBER_end >= 1. || p.QBER_begin >= p.QBER_end)
                throw std::runtime_error("Invalid QBER begin or end parameters. QBER must be: 0 < QBER < 1, and begin must be less than end.");
            if (p.QBER_step <= 0.)
                throw std::runtime_error("QBER step must be > 0!");
            const double epsilon = 1e-6;
            if (p.QBER_step - epsilon > p.QBER_end - p.QBER_begin)
                throw std::runtime_error("QBER step is too large.");
        }
        std::sort(cfg.R_QBER_PARAMETERS.begin(), cfg.R_QBER_PARAMETERS.end(),
                  [](const R_QBER_params &a, const R_QBER_params &b) { return a.code_rate < b.code_rate; });

        // optional keys of this implementation
        if (root.contains("device_precision"))
        {
            cfg.DEVICE_PRECISION = static_cast<int>(root.at("device_precision").as_size());
            if (cfg.DEVICE_PRECISION != 64 && cfg.DEVICE_PRECISION != 32)
                throw std::runtime_error("device_precision must be 64 or 32!");
        }
        if (root.contains("device_fp32_fast_math"))
            cfg.DEVICE_FP32_FAST = root.at("device_fp32_fast_math").as_bool();
        if (root.contains("device_fp64_fused_ratio"))
            cfg.DEVICE_FP64_FUSED = root.at("device_fp64_fused_ratio").as_bool();
        if (root.contains("device_gpus"))
            cfg.DEVICE_GPUS = static_cast<int>(root.at("device_gpus").as_size());
        if (root.contains("device_force_allreduce"))
            cfg.DEVICE_FORCE_ALLREDUCE = root.at("device_force_allreduce").as_bool();
        if (root.contains("device_batch_frames"))
        {
            cfg.DEVICE_BATCH_FRAMES = root.at("device_batch_frames").as_size();
            if (cfg.DEVICE_BATCH_FRAMES < 1)
                throw std::runtime_error("device_batch_frames must be >= 1!");
        }
        return cfg;
    }
    catch (const std::exception &)
    {
        std::cerr << "An error occurred while reading a configuration parameter.\n";
        throw;
    }
}
