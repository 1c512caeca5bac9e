// Batch-mode entry point, the counterpart of the reference's src/main.cpp:15-68: reads <dir>/config.json, every matrix
// in <dir>/alist_sparse_matrices (or dense_matrices), runs the sweep on the GPUs and writes <dir>/results/*.csv.
// <dir> is argv[1], else $QKD_SOURCE_DIR, else the compile-time SOURCE_DIR, else ".".
#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <iostream>
#include <string>

#include "qkd_ldpc.hpp"
#include "trace_print.hpp"

config_data CFG;

std::vector<fs::path> get_file_paths_in_directory(const fs::path &directory_path)
{
    std::vector<fs::path> files;
    try
    {
        if (!fs::exists(directory_path) || !fs::is_directory(directory_path))
            throw std::runtime_error("Directory doesn't exist.");
        for (const auto &entry : fs::directory_iterator(directory_path))
            if (fs::is_regular_file(entry.path()))
                files.push_back(entry.path());
    }
    catch (const std::exception &)
    {
        std::cerr << "An error occurred while getting file paths in directory: " << directory_path.string() << "\n";
        throw;
    }
    return files;
}

// Inspection modes used by the test-suite (no GPU needed):
//   --dump-matrix <alist|dense> <file>   prints the loaded H_matrix
//   --time-load <alist|dense> <file>     loads the file, prints seconds, N, M, edges and a checksum of both adjacency halves
//   --gen <seed> <n> <qber>              prints the exact QBER and Alice's / Bob's keys of one trial
//   --seeds <seed> <count>               prints raw xoshiro256++ outputs
//   --peg <n> <m> <dv> <seed> <out> [lim] writes a seeded PEG code as alist (configs[3], configs[4] of BASELINE.json)
//   --rate-split <n> <m> <qber> <delta> <f>  prints the punctured and shortened counts of device_rate_adaptation at that point
static int inspect(int argc, char **argv)
{
    const std::string mode = argv[1];
    if (mode == "--dump-matrix" && argc == 4)
    {
        H_matrix h;
        if (std::string(argv[2]) == "dense")
            read_dense_matrix(argv[3], h);
        else
            read_sparse_alist_matrix(argv[3], h);
        std::cout << h.num_bit_nodes << " " << h.num_check_nodes << " " << h.max_bit_nodes_weight << " " << h.max_check_nodes_weight << " "
                  << (h.is_regular ? 1 : 0) << "\n";
        for (size_t i = 0; i < h.num_bit_nodes; ++i)
        {
            std::cout << h.bit_nodes_weight[i];
            for (int k = 0; k < h.bit_nodes_weight[i]; ++k)
                std::cout << " " << h.bit_nodes[i][k];
            std::cout << "\n";
        }
        for (size_t j = 0; j < h.num_check_nodes; ++j)
        {
            std::cout << h.check_nodes_weight[j];
            for (int k = 0; k < h.check_nodes_weight[j]; ++k)
                std::cout << " " << h.check_nodes[j][k];
            std::cout << "\n";
        }
        free_matrix_H(h);
        return EXIT_SUCCESS;
    }
    if (mode == "--time-load" && argc == 4)
    {
        const auto t0 = std::chrono::steady_clock::now();
        H_matrix h;
        if (std::string(argv[2]) == "dense")
            read_dense_matrix(argv[3], h);
        else
            read_sparse_alist_matrix(argv[3], h);
        const double seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        unsigned long long edges = 0, sum_bits = 0, sum_checks = 0;
        for (size_t i = 0; i < h.num_bit_nodes; ++i)
            for (int k = 0; k < h.bit_nodes_weight[i]; ++k, ++edges)
                sum_bits += static_cast<unsigned long long>(h.bit_nodes[i][k]) * (i + 1);
        for (size_t j = 0; j < h.num_check_nodes; ++j)
            for (int k = 0; k < h.check_nodes_weight[j]; ++k)
                sum_checks += static_cast<unsigned long long>(h.check_nodes[j][k] + 1) * j;
        std::cout << seconds << " " << h.num_bit_nodes << " " << h.num_check_nodes << " " << edges << " " << sum_bits << " " << sum_checks << "\n";
        free_matrix_H(h);
        return EXIT_SUCCESS;
    }
    if (mode == "--gen" && argc == 5)
    {
        const size_t seed = std::strtoull(argv[2], nullptr, 10), n = std::strtoull(argv[3], nullptr, 10);
        const double q = std::strtod(argv[4], nullptr);
        XoshiroCpp::Xoshiro256PlusPlus prng(seed);
        std::vector<int> a(n), b(n);
        generate_random_bit_array(prng, n, a.data());
        const double exact = introduce_errors(prng, a.data(), n, q, b.data());
        std::cout.precision(17);
        std::cout << exact << "\n";
        for (int v : a)
            std::cout << v;
        std::cout << "\n";
        for (int v : b)
            std::cout << v;
        std::cout << "\n";
        return EXIT_SUCCESS;
    }
    if (mode == "--seeds" && argc == 4)
    {
        XoshiroCpp::Xoshiro256PlusPlus prng(std::strtoull(argv[2], nullptr, 10));
        for (size_t i = 0, k = std::strtoull(argv[3], nullptr, 10); i < k; ++i)
            std::cout << prng() << "\n";
        return EXIT_SUCCESS;
    }
    if (mode == "--peg" && (argc == 7 || argc == 8))
    {
        qkd_b200::generate_peg_alist(std::strtoull(argv[2], nullptr, 10), std::strtoull(argv[3], nullptr, 10), std::strtoull(argv[4], nullptr, 10),
                                     std::strtoull(argv[5], nullptr, 10), argc == 8 ? std::strtoull(argv[7], nullptr, 10) : 4096, argv[6]);
        return EXIT_SUCCESS;
    }
    if (mode == "--rate-split" && argc == 7)
    {
        const auto [p, s] = qkd_b200::rate_split(std::strtoull(argv[2], nullptr, 10), std::strtoull(argv[3], nullptr, 10), std::strtod(argv[4], nullptr),
                                                 std::strtod(argv[5], nullptr), std::strtod(argv[6], nullptr));
        std::cout << p << " " << s << "\n";
        return EXIT_SUCCESS;
    }
    std::cerr << "usage: qkd_ldpc_b200_sim [dir] | --peg <n> <m> <col_weight> <seed> <out.alist> [bfs_limit] | --dump-matrix <alist|dense> <file> | --time-load <alist|dense> <file> | --gen <seed> <n> <qber> | --seeds <seed> <count> | --rate-split <n> <m> <qber> <delta> <f>\n";
    return EXIT_FAILURE;
}

int main(int argc, char **argv)
{
    if (argc > 1 && std::string(argv[1]).rfind("--", 0) == 0)
    {
        try
        {
            return inspect(argc, argv);
        }
        catch (const std::exception &e)
        {
            std::cerr << "ERROR: " << e.what() << "\n";
            return EXIT_FAILURE;
        }
    }
#ifndef SOURCE_DIR
#define SOURCE_DIR "."
#endif
    const char *env = std::getenv("QKD_SOURCE_DIR");
    const fs::path root = argc > 1 ? fs::path(argv[1]) : (env ? fs::path(env) : fs::path(SOURCE_DIR));
    std::vector<sim_input> sim_inputs;
    try
    {
        CFG = get_config_data(root / "config.json");
        const fs::path matrix_dir = root / (CFG.USE_DENSE_MATRICES ? "dense_matrices" : "alist_sparse_matrices");
        if (CFG.INTERACTIVE_MODE)
        {
            qkd_b200::print_coloured(qkd_b200::colour::purple, "INTERACTIVE MODE\n");
            QKD_LDPC_interactive_simulation(matrix_dir);
            qkd_b200::release_device_state();
            return EXIT_SUCCESS;
        }
        qkd_b200::print_coloured(qkd_b200::colour::purple, "BATCH MODE\n");
        std::fflush(stdout);
        const std::vector<fs::path> matrix_paths = get_file_paths_in_directory(matrix_dir);
        if (matrix_paths.empty())
            throw std::runtime_error("Matrix folder is empty: " + matrix_dir.string());
        sim_inputs.resize(matrix_paths.size());
        prepare_sim_inputs(matrix_paths, sim_inputs);
        qkd_b200::set_progress_directory(root / "results");
        const std::vector<sim_result> results = QKD_LDPC_batch_simulation(sim_inputs);
        for (sim_input &in : sim_inputs)
            free_matrix_H(in.matrix);
        sim_inputs.clear();
        std::cout << "The results will be written to the directory: " << (root / "results").string() << "\n";
        write_file(results, root / "results");
        qkd_b200::write_report(qkd_b200::last_sweep_report(), root / "results");
        const auto &rep = qkd_b200::last_sweep_report();
        std::cout << "frames " << rep.frames << ", frame-iterations " << rep.frame_iterations << ", " << rep.gpus << " GPU(s), " << rep.seconds_total
                  << " s total (" << rep.seconds_startup << " s start-up = CUDA contexts beside " << rep.seconds_comm_setup << " s of NCCL communicator set-up; " << rep.seconds_device
                  << " s in device calls per worker, " << rep.seconds_reduce << " s all-reduce): "
                  << rep.frames / rep.seconds_total << " frames/s overall, " << rep.frames / std::max(1e-9, rep.seconds_total - rep.seconds_startup)
                  << " frames/s once the GPUs are up\n";
    }
    catch (const std::exception &e)
    {
        for (sim_input &in : sim_inputs)
            free_matrix_H(in.matrix);
        std::cerr << "ERROR: " << e.what() << "\n";
        qkd_b200::release_device_state();
        return EXIT_FAILURE;
    }
    qkd_b200::release_device_state();
    return EXIT_SUCCESS;
}
