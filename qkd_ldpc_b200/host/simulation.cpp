// The config.json-driven QBER sweep as a frame-batch scheduler.
//
// Mirrors the reference's src/simulation.cpp: write_file :4-44, get_rate_based_QBER_range :48-70, prepare_sim_inputs
// :140-158, run_trial :161-189, QKD_LDPC_batch_simulation :192-316 -- same signatures, same trial seeds
// (seeds[k] + index of the (matrix, QBER) point), same statistics, same CSV. What changes is the execution model: instead
// of one pool task per trial that generates AND decodes on a CPU core, the trials are cut into batches, and each batch is
// one qlb_run_trials call that draws the keys on a GPU from the trial seeds (bit-exact with the reference's generator) and
// reconciles them. Trials are independent, so batches are dealt to all GPUs of the box with no exchange while decoding;
// per-point statistics are integer histograms, summed over the GPUs by one NCCL all-reduce per sweep (qlb_stats_allreduce).
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cmath>
#include <condition_variable>
#include <fstream>
#include <iostream>
#include <limits>
#include <sstream>
#include <algorithm>
#include <mutex>
#include <random>
#include <stdexcept>
#include <thread>
#include <tuple>

#include "device_bridge.hpp"
#include "qkd_ldpc.hpp"
#include "trace_print.hpp"

namespace
{
    qkd_b200::sweep_report g_report;

    // One batch of the sweep: `frames` trials of one point, seeds[first_trial ...] + point (src/simulation.cpp:247).
    struct batch
    {
        size_t point, first_trial, frames;
    };

    [[noreturn]] void key_too_small(size_t n) { throw std::runtime_error("Key size '" + std::to_string(n) + "' is too small for QBER."); }

    // Header and row of the side file (qkd_b200::write_report); the last four columns exist with rate adaptation only.
    std::string report_header()
    {
        return std::string("SIM;MATRIX_FILENAME;M;N;QBER;FRAMES;SECONDS;FRAMES_PER_S;SIFTED_MBIT_PER_S;FRAME_ITERATIONS;MEAN_ITERATIONS;"
                           "EFFICIENCY_F;LEAKED_BITS_PER_FRAME;GPUS;PRECISION") +
               (CFG.DEVICE_RATE_ADAPTATION ? ";PUNCTURED;SHORTENED;KEY_BITS;EFFECTIVE_RATE\n" : "\n");
    }
    std::string report_row(const qkd_b200::point_report &p, int gpus)
    {
        std::ostringstream out;
        const std::string precision = CFG.DEVICE_PRECISION == 32 ? (CFG.DEVICE_FP32_FAST ? "fp32-fast" : CFG.DEVICE_FP32_MIN_SUM_SCALE != 0. ? "fp32-min-sum" : "fp32") : (CFG.DEVICE_FP64_FUSED ? "fp64-fused" : "fp64");
        const double q = p.exact_qber, h2 = -q * std::log2(q) - (1. - q) * std::log2(1. - q);
        const double fps = p.seconds > 0 ? p.frames / p.seconds : 0.;
        // key bits and leaked bits per frame: N and M with plain syndrome coding
        const size_t key_bits = p.num_bit_nodes - p.punctured - p.shortened, leak = p.num_check_nodes - p.punctured;
        out << p.sim_number << ";" << p.matrix_filename << ";" << p.num_check_nodes << ";" << p.num_bit_nodes << ";" << q << ";" << p.frames << ";"
            << p.seconds << ";" << fps << ";" << fps * key_bits / 1e6 << ";" << p.frame_iterations << ";"
            << static_cast<double>(p.frame_iterations) / p.frames << ";" << (static_cast<double>(leak) / key_bits) / h2 << ";"
            << leak << ";" << gpus << ";" << precision;
        if (CFG.DEVICE_RATE_ADAPTATION)
            out << ";" << p.punctured << ";" << p.shortened << ";" << key_bits << ";"
                << static_cast<double>(p.num_bit_nodes - p.num_check_nodes - p.shortened) / key_bits;
        out << "\n";
        return out.str();
    }
}

namespace qkd_b200
{
    const sweep_report &last_sweep_report() { return g_report; }

    std::pair<size_t, size_t> rate_split(size_t n, size_t m, double q, double delta, double target_efficiency)
    {
        const double h2 = -q * std::log2(q) - (1. - q) * std::log2(1. - q), r0 = 1. - static_cast<double>(m) / n;
        const long long d = std::llround(delta * n);
        const long long s = std::clamp(std::llround((r0 - (1. - target_efficiency * h2) * (1. - delta)) * n), 0LL, d);
        return {static_cast<size_t>(d - s), static_cast<size_t>(s)};
    }

    void write_report(const sweep_report &report, fs::path directory)
    {
        if (!fs::exists(directory))
            fs::create_directories(directory);
        const std::string stem = "throughput(trial_num=" + std::to_string(CFG.TRIALS_NUMBER) + ",max_sum_prod_iters=" +
                                 std::to_string(CFG.SUM_PRODUCT_MAX_ITERATIONS) + ",seed=" + std::to_string(CFG.SIMULATION_SEED) + ")";
        fs::path target = directory / (stem + ".csv");
        for (size_t dup = 1; fs::exists(target); ++dup)
            target = directory / (stem + "_" + std::to_string(dup) + ".csv");
        std::ofstream out(target, std::ios::out | std::ios::trunc);
        out << report_header();
        for (const point_report &p : report.points)
            out << report_row(p, report.gpus);
    }

    std::vector<std::string> matrix_warnings(const H_matrix &h)
    {
        std::vector<std::string> w;
        size_t unsorted_bits = 0, unsorted_checks = 0, dup = 0;
        for (size_t i = 0; i < h.num_bit_nodes; ++i)
            for (int k = 1; k < h.bit_nodes_weight[i]; ++k)
            {
                unsorted_bits += h.bit_nodes[i][k] < h.bit_nodes[i][k - 1];
                dup += h.bit_nodes[i][k] == h.bit_nodes[i][k - 1];
            }
        for (size_t j = 0; j < h.num_check_nodes; ++j)
            for (int k = 1; k < h.check_nodes_weight[j]; ++k)
                unsorted_checks += h.check_nodes[j][k] < h.check_nodes[j][k - 1];
        if (unsorted_bits || unsorted_checks)
            w.push_back("adjacency lists are not sorted ascending (" + std::to_string(unsorted_bits) + " bit-list and " + std::to_string(unsorted_checks) +
                        " check-list inversions): the reference routes messages by arrival order, which is only the intended routing for sorted lists");
        if (dup)
            w.push_back(std::to_string(dup) + " duplicate entries in the bit lists (a double edge cancels in the syndrome but not in the decoder)");
        return w;
    }
}

// CSV, byte for byte the reference's format (default ostream precision, ';' separated, FER = 1 - ratio_ldpc).
void write_file(const std::vector<sim_result> &data, fs::path directory)
{
    try
    {
        if (!fs::exists(directory))
            fs::create_directories(directory);
        const std::string stem = "ldpc(trial_num=" + std::to_string(CFG.TRIALS_NUMBER) + ",max_sum_prod_iters=" +
                                 std::to_string(CFG.SUM_PRODUCT_MAX_ITERATIONS) + ",seed=" + std::to_string(CFG.SIMULATION_SEED) + ")";
        fs::path target = directory / (stem + ".csv");
        for (size_t dup = 1; fs::exists(target); ++dup)
            target = directory / (stem + "_" + std::to_string(dup) + ".csv");

        std::ofstream out(target, std::ios::out | std::ios::trunc);
        out << "№;MATRIX_FILENAME;TYPE;CODE_RATE;M;N;QBER;ITERATIONS_SUCCESSFUL_SP_MEAN;ITERATIONS_SUCCESSFUL_SP_STD_DEV;"
               "ITERATIONS_SUCCESSFUL_SP_MIN;ITERATIONS_SUCCESSFUL_SP_MAX;RATIO_TRIALS_SUCCESSFUL_SP;RATIO_TRIALS_SUCCESSFUL_LDPC;FER\n";
        for (const sim_result &r : data)
            out << r.sim_number << ";" << r.matrix_filename << ";" << (r.is_regular ? "regular" : "irregular") << ";"
                << 1. - (static_cast<double>(r.num_check_nodes) / r.num_bit_nodes) << ";" << r.num_check_nodes << ";" << r.num_bit_nodes << ";"
                << r.initial_QBER << ";" << r.iterations_successful_sp_mean << ";" << r.iterations_successful_sp_std_dev << ";"
                << r.iterations_successful_sp_min << ";" << r.iterations_successful_sp_max << ";" << r.ratio_trials_successful_sp << ";"
                << r.ratio_trials_successful_ldpc << ";" << 1. - r.ratio_trials_successful_ldpc << "\n";
    }
    catch (const std::exception &)
    {
        std::cerr << "An error occurred while writing to the file.\n";
        throw;
    }
}

// First preset (sorted by rate) whose code_rate is >= the matrix's; end-exclusive grid begin + j*step, j < round((end-begin)/step).
std::vector<double> get_rate_based_QBER_range(const double code_rate, const std::vector<R_QBER_params> &R_QBER_parameters)
{
    for (const R_QBER_params &p : R_QBER_parameters)
    {
        if (code_rate > p.code_rate)
            continue;
        const size_t steps = round((p.QBER_end - p.QBER_begin) / p.QBER_step);
        std::vector<double> grid;
        for (size_t j = 0; j < steps; ++j)
            grid.push_back(p.QBER_begin + j * p.QBER_step);
        if (!grid.empty())
            return grid;
        break;
    }
    throw std::runtime_error("An error occurred when generating a QBER range based on code rate.");
}

void prepare_sim_inputs(const std::vector<fs::path> &matrix_paths, std::vector<sim_input> &sim_inputs_out)
{
    for (size_t i = 0; i < matrix_paths.size(); ++i)
    {
        sim_input &in = sim_inputs_out[i];
        if (CFG.USE_DENSE_MATRICES)
            read_dense_matrix(matrix_paths[i], in.matrix);
        else
            read_sparse_alist_matrix(matrix_paths[i], in.matrix);
        in.matrix_path = matrix_paths[i];
        for (const std::string &warning : qkd_b200::matrix_warnings(in.matrix))
            std::cerr << "WARNING (" << matrix_paths[i].filename().string() << "): " << warning << "\n";
        if (!CFG.INTERACTIVE_MODE)
            qkd_b200::code_for(in.matrix); // a matrix the device layout rejects must stop the run here, before any GPU work
        const double code_rate = 1. - (static_cast<double>(in.matrix.num_check_nodes) / in.matrix.num_bit_nodes);
        in.QBER = get_rate_based_QBER_range(code_rate, CFG.R_QBER_PARAMETERS);
    }
}

// One frame per QBER value of the matrix picked on stdin, printed step by step: the reference's interactive mode
// (src/simulation.cpp:73-137, src/utils.cpp:50-67), each frame decoded on the GPU.
fs::path select_matrix_file(const std::vector<fs::path> &matrix_paths)
{
    using qkd_b200::colour;
    qkd_b200::print_coloured(colour::green, "Choose file: \n");
    for (size_t i = 0; i < matrix_paths.size(); i++)
        qkd_b200::print_coloured(colour::green, std::to_string(i + 1) + ". " + matrix_paths[i].filename().string() + "\n");
    std::fflush(stdout);
    int file_index = 0;
    std::cin >> file_index;
    file_index -= 1;
    if (file_index < 0 || file_index >= static_cast<int>(matrix_paths.size()))
        throw std::runtime_error("Wrong file number.");
    return matrix_paths[file_index];
}

void QKD_LDPC_interactive_simulation(fs::path matrix_dir_path)
{
    using qkd_b200::colour;
    using qkd_b200::print_coloured;
    H_matrix matrix;
    const std::vector<fs::path> matrix_paths = get_file_paths_in_directory(matrix_dir_path);
    const fs::path matrix_path = select_matrix_file(matrix_paths);
    if (CFG.USE_DENSE_MATRICES)
        read_dense_matrix(matrix_path, matrix);
    else
        read_sparse_alist_matrix(matrix_path, matrix);
    try
    {
        print_coloured(colour::green, std::string(matrix.is_regular ? "Matrix H is regular." : "Matrix H is irregular.") + "\n");
        const size_t n = matrix.num_bit_nodes;
        std::vector<int> alice(n), bob(n);
        XoshiroCpp::Xoshiro256PlusPlus prng(CFG.SIMULATION_SEED); // one stream for all frames, as in the reference (:95)
        const double code_rate = 1. - (static_cast<double>(matrix.num_check_nodes) / matrix.num_bit_nodes);
        const std::vector<double> QBER = get_rate_based_QBER_range(code_rate, CFG.R_QBER_PARAMETERS);
        for (size_t i = 0; i < QBER.size(); i++)
        {
            print_coloured(colour::green, "\u2116:" + std::to_string(i + 1) + "\n");
            generate_random_bit_array(prng, n, alice.data());
            const double initial_QBER = introduce_errors(prng, alice.data(), n, QBER[i], bob.data());
            print_coloured(colour::green, "Actual QBER: " + qkd_b200::format_shortest(initial_QBER) + "\n");
            if (initial_QBER == 0.)
                key_too_small(n);
            int error_num = 0;
            for (size_t k = 0; k < n; k++)
                error_num += alice[k] ^ bob[k];
            print_coloured(colour::green, "Number of errors in a key: " + std::to_string(error_num) + "\n");
            std::fflush(stdout);
            const LDPC_result r = matrix.is_regular ? QKD_LDPC_regular(alice.data(), bob.data(), initial_QBER, matrix)
                                                    : QKD_LDPC_irregular(alice.data(), bob.data(), initial_QBER, matrix);
            print_coloured(colour::green, "Iterations performed: " + std::to_string(r.sp_res.iterations_num) + "\n");
            print_coloured(colour::green, std::string(r.keys_match && r.sp_res.syndromes_match ? "Error reconciliation SUCCESSFUL" : "Error reconciliation FAILED") + "\n\n");
            std::fflush(stdout);
        }
    }
    catch (...)
    {
        free_matrix_H(matrix);
        throw;
    }
    free_matrix_H(matrix);
}

// A single trial (batch of one). Throws like the reference when floor(N * QBER) == 0.
trial_result run_trial(const H_matrix &matrix, const double QBER, size_t seed)
{
    const size_t n = matrix.num_bit_nodes;
    XoshiroCpp::Xoshiro256PlusPlus prng(seed);
    std::vector<int> alice(n), bob(n);
    trial_result result;
    generate_random_bit_array(prng, n, alice.data());
    result.initial_QBER = introduce_errors(prng, alice.data(), n, QBER, bob.data());
    if (result.initial_QBER == 0.)
        key_too_small(n);
    result.ldpc_res = matrix.is_regular ? QKD_LDPC_regular(alice.data(), bob.data(), result.initial_QBER, matrix)
                                        : QKD_LDPC_irregular(alice.data(), bob.data(), result.initial_QBER, matrix);
    return result;
}

namespace
{
    // Integer statistics of one (matrix, QBER) point: histogram of iterations_num over the frames whose syndromes match, then
    // {n_sp, n_ldpc, n_trials, sum of iterations}. Everything the reference accumulates per point (src/simulation.cpp:252-312) is a
    // function of these integers, so the sums over workers / GPUs do not depend on who decoded what, nor on the reduction order.
    struct point_stats_view
    {
        const uint64_t *v;
        size_t max_it;
        uint64_t n_sp() const { return v[max_it + 1]; }
        uint64_t n_ldpc() const { return v[max_it + 2]; }
        uint64_t n_trials() const { return v[max_it + 3]; }
        uint64_t iterations() const { return v[max_it + 4]; }
    };

    // src/simulation.cpp:252-312 from the histogram: count / min / max / mean / population std-dev over the successful frames.
    // The mean is a sum of integers (exact in double, as the reference's running sum is); the std-dev sums (it - mean)^2 per
    // iteration count instead of per trial -- the same real number, rounded differently far below the CSV's six digits.
    void fill_result(sim_result &r, const point_stats_view &st, size_t trials)
    {
        const size_t max_it = st.max_it;
        size_t it_max = 0, it_min = max_it;
        double mean = 0, sd = 0;
        if (st.n_sp() > 0)
        {
            uint64_t sum = 0;
            for (size_t it = 0; it <= max_it; ++it)
                if (st.v[it])
                {
                    sum += st.v[it] * it;
                    it_max = std::max(it_max, it);
                    it_min = std::min(it_min, it);
                }
            mean = static_cast<double>(sum) / static_cast<double>(st.n_sp());
            for (size_t it = 0; it <= max_it; ++it)
                if (st.v[it])
                    sd += static_cast<double>(st.v[it]) * pow(static_cast<double>(it) - mean, 2);
            sd = sqrt(sd / static_cast<double>(st.n_sp()));
        }
        r.iterations_successful_sp_max = it_max;
        r.iterations_successful_sp_min = (it_min == max_it) ? 0 : it_min; // :306
        r.iterations_successful_sp_mean = mean;
        r.iterations_successful_sp_std_dev = sd;
        r.ratio_trials_successful_ldpc = static_cast<double>(st.n_ldpc()) / trials;
        r.ratio_trials_successful_sp = static_cast<double>(st.n_sp()) / trials;
    }

    fs::path g_progress_dir; // where finished points are appended while the sweep runs (empty: nowhere)

    std::string csv_row(const sim_result &r)
    {
        std::ostringstream out;
        out << r.sim_number << ";" << r.matrix_filename << ";" << (r.is_regular ? "regular" : "irregular") << ";"
            << 1. - (static_cast<double>(r.num_check_nodes) / r.num_bit_nodes) << ";" << r.num_check_nodes << ";" << r.num_bit_nodes << ";"
            << r.initial_QBER << ";" << r.iterations_successful_sp_mean << ";" << r.iterations_successful_sp_std_dev << ";"
            << r.iterations_successful_sp_min << ";" << r.iterations_successful_sp_max << ";" << r.ratio_trials_successful_sp << ";"
            << r.ratio_trials_successful_ldpc << ";" << 1. - r.ratio_trials_successful_ldpc << "\n";
        return out.str();
    }
    const char *kCsvHeader = "№;MATRIX_FILENAME;TYPE;CODE_RATE;M;N;QBER;ITERATIONS_SUCCESSFUL_SP_MEAN;ITERATIONS_SUCCESSFUL_SP_STD_DEV;"
                             "ITERATIONS_SUCCESSFUL_SP_MIN;ITERATIONS_SUCCESSFUL_SP_MAX;RATIO_TRIALS_SUCCESSFUL_SP;RATIO_TRIALS_SUCCESSFUL_LDPC;FER\n";
}

namespace qkd_b200
{
    void set_progress_directory(const fs::path &directory) { g_progress_dir = directory; }
}

// The frame-batch scheduler. Every (point, block of trials) is an independent batch; ALL batches of the sweep are listed up
// front -- there is no barrier between QBER points -- and claimed in that order by two host threads per GPU, each with a
// context (stream + staging buffers) of its own. Workers accumulate integer statistics per point; a finished point is
// appended to the progress files at once (nothing is held per trial, nothing is lost on abort). The statistics of the
// returned results come from the sweep's ONE collective: a SUM all-reduce over the GPUs of the [points x (max_it + 5)] integers (qlb_stats_allreduce, NCCL).
std::vector<sim_result> QKD_LDPC_batch_simulation(const std::vector<sim_input> &sim_in)
{
    using clock = std::chrono::steady_clock;
    const auto t_start = clock::now();
    auto seconds_since = [](clock::time_point t0) { return std::chrono::duration<double>(clock::now() - t0).count(); };
    const size_t trials = CFG.TRIALS_NUMBER;
    const size_t max_it = CFG.SUM_PRODUCT_MAX_ITERATIONS;
    const size_t stats_width = max_it + 1 + 4;

    // seeds[k]: the k-th raw output of xoshiro256++(SIMULATION_SEED), drawn the way the reference draws them (:222-228)
    XoshiroCpp::Xoshiro256PlusPlus seed_prng(CFG.SIMULATION_SEED);
    std::uniform_int_distribution<size_t> any_size(0, std::numeric_limits<size_t>::max());
    std::vector<size_t> seeds(trials);
    for (size_t &s : seeds)
        s = any_size(seed_prng);

    // ---- the points of the sweep, numbered as the reference numbers them (curr_sim, :231-236, 312) ------------------------
    struct point
    {
        const sim_input *in;
        double qber, exact_qber;
        qlb_code *code;
        size_t punctured = 0, shortened = 0;
        std::vector<uint8_t> pos_class; // rate adaptation: qlb_rate_pattern of the point (empty without it)
        std::atomic<size_t> batches_left{0};
        std::atomic<uint64_t> device_ns{0};
    };
    size_t points_total = 0;
    for (const sim_input &in : sim_in)
        points_total += in.QBER.size();
    std::vector<point> points(points_total);
    {
        size_t pt = 0;
        for (const sim_input &in : sim_in)
            for (const double q : in.QBER)
            {
                point &p = points[pt];
                p.code = qkd_b200::code_for(in.matrix);
                if (CFG.DEVICE_RATE_ADAPTATION)
                {
                    std::tie(p.punctured, p.shortened) = qkd_b200::rate_split(in.matrix.num_bit_nodes, in.matrix.num_check_nodes, q, CFG.DEVICE_RATE_MODULATED_FRACTION,
                                                                              CFG.DEVICE_RATE_TARGET_EFFICIENCY);
                    if (p.punctured > 0 && (CFG.DEVICE_PRECISION != 32 || CFG.DEVICE_FP32_FAST))
                        throw std::runtime_error("device_rate_adaptation punctures " + std::to_string(p.punctured) + " bits at QBER " + std::to_string(q) +
                                                 ": puncturing needs device_precision 32 without device_fp32_fast_math (fp32 or fp32 min-sum)!");
                    if (p.shortened > 0 && !CFG.ENABLE_SUM_PRODUCT_MSG_LLR_THRESHOLD)
                        throw std::runtime_error("device_rate_adaptation shortens " + std::to_string(p.shortened) + " bits at QBER " + std::to_string(q) +
                                                 ": shortening needs enable_sum_product_msg_llr_threshold!");
                    p.pos_class.resize(in.matrix.num_bit_nodes);
                    if (qlb_rate_pattern(p.code, static_cast<int32_t>(p.punctured), static_cast<int32_t>(p.shortened), CFG.DEVICE_RATE_PATTERN_SEED,
                                         p.pos_class.data()) != QLB_OK)
                        throw std::runtime_error(std::string("device_rate_adaptation: ") + qlb_last_error());
                }
                const size_t n = in.matrix.num_bit_nodes - p.punctured - p.shortened; // the key bits of a frame
                if (static_cast<size_t>(n * q) == 0)
                    key_too_small(n); // the reference throws from inside the point's first trial (src/simulation.cpp:170-175)
                p.in = &in;
                p.qber = q;
                p.exact_qber = static_cast<double>(static_cast<size_t>(n * q)) / n; // introduce_errors' return value (:436-459)
                ++pt;
            }
    }

    int gpus = qkd_b200::usable_devices();
    if (gpus < 1)
        throw std::runtime_error("no CUDA device is available: this build has no CPU decoder");
    if (CFG.DEVICE_GPUS > 0)
        gpus = std::min(gpus, CFG.DEVICE_GPUS);
    const qlb_decode_params params = qkd_b200::params_from_cfg(max_it, CFG.SUM_PRODUCT_MSG_LLR_THRESHOLD);
    g_report = qkd_b200::sweep_report{};
    std::vector<sim_result> sim_results(points_total);
    for (size_t pt = 0; pt < points_total; ++pt)
    {
        const H_matrix &h = points[pt].in->matrix;
        sim_result &r = sim_results[pt];
        r.sim_number = pt;
        r.matrix_filename = points[pt].in->matrix_path.filename().string();
        r.is_regular = h.is_regular;
        r.num_bit_nodes = h.num_bit_nodes;
        r.num_check_nodes = h.num_check_nodes;
        r.initial_QBER = points[pt].exact_qber; // the reference copies trial 0's (:304); every trial of a point has the same
    }
    auto report_of = [&](size_t pt, uint64_t frame_iterations, double seconds)
    {
        qkd_b200::point_report pr;
        pr.sim_number = pt;
        pr.matrix_filename = sim_results[pt].matrix_filename;
        pr.num_bit_nodes = sim_results[pt].num_bit_nodes;
        pr.num_check_nodes = sim_results[pt].num_check_nodes;
        pr.exact_qber = points[pt].exact_qber;
        pr.frames = trials;
        pr.frame_iterations = frame_iterations;
        pr.seconds = seconds;
        pr.punctured = points[pt].punctured;
        pr.shortened = points[pt].shortened;
        return pr;
    };

    // progress files: one row per finished point, flushed as it finishes; removed when the sweep completes
    std::ofstream progress_csv, progress_report;
    fs::path progress_csv_path, progress_report_path;
    if (!g_progress_dir.empty())
    {
        fs::create_directories(g_progress_dir);
        const std::string tag = "(trial_num=" + std::to_string(trials) + ",max_sum_prod_iters=" + std::to_string(max_it) + ",seed=" +
                                std::to_string(CFG.SIMULATION_SEED) + ").partial.csv";
        progress_csv_path = g_progress_dir / ("ldpc" + tag);
        progress_report_path = g_progress_dir / ("throughput" + tag);
        progress_csv.open(progress_csv_path, std::ios::out | std::ios::trunc);
        progress_report.open(progress_report_path, std::ios::out | std::ios::trunc);
        progress_csv << kCsvHeader << std::flush;
        progress_report << report_header() << std::flush;
    }
    auto flush_point = [&](size_t pt, const uint64_t *stats, double seconds)
    {
        sim_result r = sim_results[pt];
        fill_result(r, point_stats_view{stats, max_it}, trials);
        if (progress_csv.is_open())
        {
            progress_csv << csv_row(r) << std::flush;
            progress_report << report_row(report_of(pt, stats[max_it + 4], seconds), gpus) << std::flush;
        }
    };

    // With any console trace enabled the trials run one after another on this thread through run_trial, so the output reads
    // like the reference's with threads_number = 1 (its pool would interleave the prints of concurrent trials).
    const bool traced = CFG.TRACE_QKD_LDPC || CFG.TRACE_SUM_PRODUCT || CFG.TRACE_SUM_PRODUCT_LLR;
    // per GPU: [points x stats_width]; the all-reduce at the end sums them
    std::vector<std::vector<uint64_t>> gpu_stats(gpus, std::vector<uint64_t>(points_total * stats_width, 0));
    std::vector<double> point_seconds(points_total, 0.);
    double startup_seconds = 0., device_seconds = 0.;
    // NCCL communicator set-up (seconds on an 8-GPU box) starts NOW on a side thread, beside the CUDA start-up of the devices
    // that the workers are about to trigger, and the workers take their first batch only when it is done: set-up next to busy
    // GPUs was measured to take 3x longer (its device-synchronising calls queue behind the persistent decode kernels: 10.9 s
    // instead of ~3 s beside fp64 batches on 2 GPUs) and to slow the decoding by 4-15 %. So start-up = CUDA contexts + NCCL
    // communicators, in parallel; after it the GPUs only decode. The sweep's one collective runs after the workers have stopped.
    const bool reduce_over_nccl = !traced && (gpus > 1 || CFG.DEVICE_FORCE_ALLREDUCE);
    std::thread comm_thread;
    struct join_on_exit
    {
        std::thread &t;
        ~join_on_exit()
        {
            if (t.joinable())
                t.join();
        }
    } comm_joiner{comm_thread}; // an exception on the way must not destroy a running thread
    std::string comm_error;
    double comm_seconds = 0.;
    std::atomic<bool> comm_ready{!reduce_over_nccl};
    std::mutex comm_mu;
    std::condition_variable comm_cv;
    if (reduce_over_nccl)
        comm_thread = std::thread([&]
                                  {
            const auto t0 = clock::now();
            std::vector<int32_t> devices(gpus);
            for (int g = 0; g < gpus; ++g)
                devices[g] = g;
            if (qlb_stats_comm_prepare(devices.data(), gpus) != QLB_OK)
                comm_error = qlb_last_error();
            comm_seconds = seconds_since(t0);
            {
                std::lock_guard<std::mutex> lk(comm_mu);
                comm_ready = true;
            }
            comm_cv.notify_all(); });

    if (traced)
    {
        for (size_t pt = 0; pt < points_total; ++pt)
        {
            const auto t0 = clock::now();
            uint64_t *st = gpu_stats[0].data() + pt * stats_width;
            for (size_t k = 0; k < trials; ++k)
            {
                const trial_result tr = run_trial(points[pt].in->matrix, points[pt].qber, seeds[k] + pt);
                const size_t it = tr.ldpc_res.sp_res.iterations_num;
                if (tr.ldpc_res.sp_res.syndromes_match)
                {
                    ++st[std::min<size_t>(it, max_it)];
                    ++st[max_it + 1];
                    st[max_it + 2] += tr.ldpc_res.keys_match;
                }
                ++st[max_it + 3];
                st[max_it + 4] += it;
            }
            point_seconds[pt] = seconds_since(t0);
            flush_point(pt, st, point_seconds[pt]);
        }
    }
    else
    {
        // ---- batches ----------------------------------------------------------------------------------------------------
        const int workers_per_gpu = 2, workers = gpus * workers_per_gpu;
        const size_t batch_cap = std::max<size_t>(1, CFG.DEVICE_BATCH_FRAMES);
        // enough batches for every worker to get several, but none smaller than 1 024 frames (a launch fills 148 SMs)
        const size_t batch_frames = std::max<size_t>(1, std::min(batch_cap, std::max<size_t>(1024, trials * points_total / (static_cast<size_t>(workers) * 4) + 1)));
        const size_t batches_per_point = (trials + batch_frames - 1) / batch_frames;
        for (point &p : points)
            p.batches_left = batches_per_point;
        // costly points first (high QBER = many iterations): the sweep then ends on short batches, which keeps the tail of the
        // last GPU short; nothing else depends on the order
        std::vector<size_t> order(points_total);
        for (size_t pt = 0; pt < points_total; ++pt)
            order[pt] = pt;
        std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) { return points[a].qber > points[b].qber; });

        std::vector<batch> batches;
        batches.reserve(points_total * batches_per_point);
        for (const size_t pt : order)
            for (size_t first = 0; first < trials; first += batch_frames)
                batches.push_back({pt, first, std::min(batch_frames, trials - first)});
        std::atomic<size_t> next_batch{0};

        std::atomic<bool> failed{false};
        std::mutex done_mu;
        std::condition_variable done_cv;
        std::string first_error;
        auto record_error = [&](const std::string &what)
        {
            {
                std::lock_guard<std::mutex> lk(done_mu);
                if (first_error.empty())
                    first_error = what;
                failed = true;
            }
            done_cv.notify_all(); // the points still open will not finish: the main thread must stop waiting for them
        };
        std::vector<size_t> finished; // points whose last batch is done, in completion order (guarded by done_mu)
        std::atomic<int> contexts_ready{0};
        std::atomic<uint64_t> device_ns{0};
        // per worker: [points x stats_width] (no sharing while decoding), folded per GPU as points finish
        std::vector<std::vector<uint64_t>> worker_stats(workers, std::vector<uint64_t>(points_total * stats_width, 0));
        std::vector<std::thread> gpu_threads;
        for (int g = 0; g < workers; ++g)
            gpu_threads.emplace_back([&, g]
                                     {
                qlb_ctx *ctx = nullptr;
                try { ctx = qkd_b200::context(g % gpus); } // worker g drives GPU g % gpus with its own context
                catch (const std::exception &e) { record_error(e.what()); }
                {
                    std::unique_lock<std::mutex> lk(comm_mu);
                    comm_cv.wait(lk, [&] { return comm_ready.load(); });
                }
                if (++contexts_ready == workers)
                    startup_seconds = seconds_since(t_start);
                std::vector<uint32_t> iterations;
                std::vector<uint8_t> result;
                for (size_t i; !failed && (i = next_batch.fetch_add(1)) < batches.size();)
                {
                    const batch &b = batches[i];
                    point &p = points[b.point];
                    iterations.resize(b.frames);
                    result.resize(b.frames);
                    const auto t0 = clock::now();
                    double exact = 0;
                    const uint64_t *trial_seeds = reinterpret_cast<const uint64_t *>(&seeds[b.first_trial]);
                    const int rc = p.pos_class.empty()
                                       ? qlb_run_trials(ctx, p.code, &params, static_cast<int64_t>(b.frames), trial_seeds, b.point, p.qber, iterations.data(),
                                                        result.data(), &exact)
                                       : qlb_run_trials_adapted(ctx, p.code, &params, p.pos_class.data(), static_cast<int64_t>(b.frames), trial_seeds, b.point,
                                                                p.qber, iterations.data(), result.data(), &exact);
                    const uint64_t ns = std::chrono::duration_cast<std::chrono::nanoseconds>(clock::now() - t0).count();
                    device_ns += ns;
                    p.device_ns += ns;
                    if (rc != QLB_OK)
                    {
                        record_error(qlb_last_error());
                        return;
                    }
                    uint64_t *st = worker_stats[g].data() + b.point * stats_width;
                    for (size_t f = 0; f < b.frames; ++f)
                    {
                        const size_t it = iterations[f];
                        if (result[f] & QLB_RES_SYNDROMES_MATCH)
                        {
                            ++st[std::min<size_t>(it, max_it)];
                            ++st[max_it + 1];
                            st[max_it + 2] += (result[f] & QLB_RES_KEYS_MATCH) != 0;
                        }
                        ++st[max_it + 3];
                        st[max_it + 4] += it;
                    }
                    if (p.batches_left.fetch_sub(1, std::memory_order_acq_rel) == 1) // every worker's share of this point is in
                    {
                        std::lock_guard<std::mutex> lk(done_mu);
                        finished.push_back(b.point);
                        done_cv.notify_all();
                    }
                } });
        auto join_workers = [&]
        {
            for (auto &t : gpu_threads)
                t.join();
        };

        try
        {
            // ---- flush points as they finish, until every point has or a worker has failed -------------------------------
            std::unique_lock<std::mutex> lk(done_mu);
            for (size_t flushed = 0; flushed < points_total && !failed;)
            {
                done_cv.wait(lk, [&] { return flushed < finished.size() || failed.load(); });
                while (flushed < finished.size())
                {
                    const size_t pt = finished[flushed++];
                    lk.unlock();
                    for (int w = 0; w < workers; ++w)
                    {
                        const uint64_t *src = worker_stats[w].data() + pt * stats_width;
                        uint64_t *acc = gpu_stats[w % gpus].data() + pt * stats_width;
                        for (size_t x = 0; x < stats_width; ++x)
                            acc[x] += src[x];
                    }
                    std::vector<uint64_t> sum(stats_width, 0);
                    for (int g = 0; g < gpus; ++g)
                        for (size_t x = 0; x < stats_width; ++x)
                            sum[x] += gpu_stats[g][pt * stats_width + x];
                    point_seconds[pt] = points[pt].device_ns.load() * 1e-9 / workers;
                    flush_point(pt, sum.data(), point_seconds[pt]);
                    lk.lock();
                }
            }
        }
        catch (...)
        {
            failed = true; // the workers stop claiming batches
            join_workers();
            throw;
        }
        join_workers();
        if (comm_thread.joinable())
            comm_thread.join();
        if (failed)
            throw std::runtime_error(first_error);
        if (!comm_error.empty())
            throw std::runtime_error("qlb_stats_comm_prepare: " + comm_error);
        device_seconds = device_ns.load() * 1e-9 / workers;
    }

    // ---- the sweep's one collective: SUM all-reduce of [points x (max_it + 5)] integers over the GPUs of this box -----------
    // It runs here, after every worker has stopped (a collective kernel next to threads that launch persistent decode kernels is
    // the documented multi-thread deadlock pattern); the communicators are normally ready by now (side thread above).
    double reduce_seconds = 0.;
    if (reduce_over_nccl)
    {
        const auto t_reduce = clock::now();
        std::vector<qlb_ctx *> ctxs;
        std::vector<uint64_t *> ptrs;
        for (int g = 0; g < gpus; ++g)
        {
            ctxs.push_back(qkd_b200::context(g));
            ptrs.push_back(gpu_stats[g].data());
        }
        qkd_b200::check(qlb_stats_allreduce(ctxs.data(), gpus, ptrs.data(), gpu_stats[0].size()), "qlb_stats_allreduce");
        reduce_seconds = seconds_since(t_reduce);
    }
    else
        for (int g = 1; g < gpus; ++g)
            for (size_t x = 0; x < gpu_stats[0].size(); ++x)
                gpu_stats[0][x] += gpu_stats[g][x];

    // ---- results from the reduced integers ------------------------------------------------------------------------------------
    size_t frames_total = 0, iterations_total = 0;
    for (size_t pt = 0; pt < points_total; ++pt)
    {
        const uint64_t *reduced = gpu_stats[0].data() + pt * stats_width;
        if (reduced[max_it + 3] != trials)
            throw std::runtime_error("reduced statistics do not account for every trial of point " + std::to_string(pt));
        fill_result(sim_results[pt], point_stats_view{reduced, max_it}, trials);
        g_report.points.push_back(report_of(pt, reduced[max_it + 4], point_seconds[pt]));
        frames_total += trials;
        iterations_total += reduced[max_it + 4];
    }
    if (progress_csv.is_open())
    {
        progress_csv.close();
        progress_report.close();
        std::error_code ec; // the caller writes the final files (write_file, write_report); the progress copies have served
        fs::remove(progress_csv_path, ec);
        fs::remove(progress_report_path, ec);
    }
    g_report.seconds_total = seconds_since(t_start);
    g_report.seconds_device = device_seconds;
    g_report.seconds_startup = startup_seconds; // CUDA initialisation + contexts: ~1 s on a 1-GPU box, ~7 s on an 8-GPU box
    g_report.seconds_comm_setup = comm_seconds;
    g_report.seconds_reduce = reduce_seconds;
    g_report.frames = frames_total;
    g_report.frame_iterations = iterations_total;
    g_report.gpus = gpus;
    return sim_results;
}
