// Host-side C++ mirror of the reference's public interface for the reconciliation hot path, implemented on top of
// the C-ABI of libqkdldpc_b200.so (include/qkd_ldpc_b200.h). Names, argument meaning and error behaviour follow the
// reference so that its callers (src/simulation.cpp:124,128,179,183; example/qkd_ldpc_example.cpp:39) keep compiling:
//
//   struct H_matrix, free_matrix_H, read_sparse_alist_matrix, read_dense_matrix   src/array_and_matrix_operations.hpp:16-53
//   calculate_syndrome_regular / _irregular, arrays_equal                        src/array_and_matrix_operations.hpp:34,39-40
//   generate_random_bit_array, introduce_errors                                   src/array_and_matrix_operations.hpp:37-38
//   SP_result, LDPC_result, sum_product_decoding_*, QKD_LDPC_*                    src/qkd_ldpc_algorithm.hpp:14-31
//   config_data, CFG, get_config_data                                             src/config.hpp:14-67
//   sim_input, trial_result, sim_result, run_trial, QKD_LDPC_batch_simulation,
//   prepare_sim_inputs, get_rate_based_QBER_range, write_file,
//   QKD_LDPC_interactive_simulation                                               src/simulation.hpp:16-50
//   console traces under CFG.TRACE_QKD_LDPC / TRACE_SUM_PRODUCT / TRACE_SUM_PRODUCT_LLR   src/qkd_ldpc_algorithm.cpp:214-327,407-442
//
// There is no CPU decoder behind these functions: they throw std::runtime_error when no B200 is usable.
#pragma once
#include <cstddef>
#include <filesystem>
#include <string>
#include <vector>

#include "XoshiroCpp.hpp"

namespace fs = std::filesystem;

struct H_matrix
{
    int **bit_nodes = nullptr;         // bit_nodes[i][k]: k-th check of bit i
    int *bit_nodes_weight = nullptr;   // checks per bit
    int **check_nodes = nullptr;       // check_nodes[j][k]: k-th bit of check j
    int *check_nodes_weight = nullptr; // bits per check
    size_t num_bit_nodes{};
    size_t num_check_nodes{};
    size_t max_bit_nodes_weight{};
    size_t max_check_nodes_weight{};
    bool is_regular{};
};

struct SP_result
{
    size_t iterations_num{};
    bool syndromes_match{};
};

struct LDPC_result
{
    SP_result sp_res{};
    bool keys_match{};
};

struct R_QBER_params
{
    double code_rate{};
    double QBER_begin{};
    double QBER_end{};
    double QBER_step{};
};

struct config_data
{
    size_t THREADS_NUMBER{}; // required and validated as in the reference; the batch sweep runs on GPU worker threads and does not read it
    size_t TRIALS_NUMBER{};
    size_t SIMULATION_SEED{};
    bool INTERACTIVE_MODE{};
    size_t SUM_PRODUCT_MAX_ITERATIONS{};
    bool USE_DENSE_MATRICES{};
    bool TRACE_QKD_LDPC{};
    bool TRACE_SUM_PRODUCT{};
    bool TRACE_SUM_PRODUCT_LLR{};
    bool ENABLE_SUM_PRODUCT_MSG_LLR_THRESHOLD{};
    double SUM_PRODUCT_MSG_LLR_THRESHOLD{};
    std::vector<R_QBER_params> R_QBER_PARAMETERS{};

    // ---- additions of this implementation; every one defaults so that an unmodified reference config.json runs ----
    int DEVICE_PRECISION = 64;     // "device_precision": 64 (the reference's arithmetic) | 32
    bool DEVICE_FP32_FAST = false; // "device_fp32_fast_math": SFU check rule for fp32
    bool DEVICE_FP64_FUSED = false; // "device_fp64_fused_ratio": one-division form of the fp64 check rule (QLB_FLAG_F64_FUSED_RATIO)
    int DEVICE_GPUS = 0;           // "device_gpus": 0 = all visible GPUs
    size_t DEVICE_BATCH_FRAMES = 32768; // "device_batch_frames": most frames per launch handed to one GPU (the on-device key generator needs
                                        // >= 32 k trials in flight to reach its 2.2 M frames/s: 4 096 -> 0.67 M, 16 384 -> 1.83 M; scripts/gen_timing2.py)
    bool DEVICE_FORCE_ALLREDUCE = false; // "device_force_allreduce": run the statistics all-reduce through NCCL even on one GPU (tests)
};

extern config_data CFG;

struct sim_input
{
    fs::path matrix_path{};
    std::vector<double> QBER{};
    H_matrix matrix{};
};

struct trial_result
{
    LDPC_result ldpc_res{};
    double initial_QBER{};
};

struct sim_result
{
    size_t sim_number{};
    std::string matrix_filename{};
    bool is_regular{};
    size_t num_bit_nodes{};
    size_t num_check_nodes{};
    double initial_QBER{};
    size_t iterations_successful_sp_max{};
    size_t iterations_successful_sp_min{};
    double iterations_successful_sp_mean{};
    double iterations_successful_sp_std_dev{};
    double ratio_trials_successful_sp{};
    double ratio_trials_successful_ldpc{};
};

// ---- matrices -------------------------------------------------------------------------------------------------------
void free_matrix_H(H_matrix &matrix);
void read_sparse_alist_matrix(const fs::path &matrix_path, H_matrix &matrix_out);
void read_dense_matrix(const fs::path &matrix_path, H_matrix &matrix_out);

// ---- keys -----------------------------------------------------------------------------------------------------------
bool arrays_equal(const int *const array1, const int *const array2, const size_t &array_length);
void generate_random_bit_array(XoshiroCpp::Xoshiro256PlusPlus &prng, size_t length, int *const random_bit_array_out);
double introduce_errors(XoshiroCpp::Xoshiro256PlusPlus &prng, const int *const bit_array, size_t array_length, double error_probability,
                        int *const bit_array_with_errors_out);

// ---- hot path (GPU) ---------------------------------------------------------------------------------------------------
void calculate_syndrome_regular(const int *const bit_array, const H_matrix &matrix, int *const syndrome_out);
void calculate_syndrome_irregular(const int *const bit_array, const H_matrix &matrix, int *const syndrome_out);
SP_result sum_product_decoding_regular(const double *const bit_array_llr, const H_matrix &matrix, const int *const syndrome,
                                       const size_t &max_num_iterations, const double &msg_threshold, int *const bit_array_out);
SP_result sum_product_decoding_irregular(const double *const bit_array_llr, const H_matrix &matrix, const int *const syndrome,
                                         const size_t &max_num_iterations, const double &msg_threshold, int *const bit_array_out);
LDPC_result QKD_LDPC_regular(const int *const alice_bit_array, const int *const bob_bit_array, const double &QBER, const H_matrix &matrix);
LDPC_result QKD_LDPC_irregular(const int *const alice_bit_array, const int *const bob_bit_array, const double &QBER, const H_matrix &matrix);

// ---- configuration and simulation ---------------------------------------------------------------------------------------
config_data get_config_data(fs::path config_path);
std::vector<fs::path> get_file_paths_in_directory(const fs::path &directory_path);
void write_file(const std::vector<sim_result> &data, fs::path directory);
std::vector<double> get_rate_based_QBER_range(const double code_rate, const std::vector<R_QBER_params> &R_QBER_parameters);
void prepare_sim_inputs(const std::vector<fs::path> &matrix_paths, std::vector<sim_input> &sim_inputs_out);
trial_result run_trial(const H_matrix &matrix, const double QBER, size_t seed);
std::vector<sim_result> QKD_LDPC_batch_simulation(const std::vector<sim_input> &sim_in);
fs::path select_matrix_file(const std::vector<fs::path> &matrix_paths);  // src/utils.hpp:18
void QKD_LDPC_interactive_simulation(fs::path matrix_dir_path);          // src/simulation.hpp:46
// print_array / print_regular_matrix / print_irregular_matrix (src/utils.hpp:15-46) live in trace_print.hpp

// ---- implementation hooks (not in the reference) -----------------------------------------------------------------------
namespace qkd_b200
{
    struct point_report // one (matrix, QBER) point of the last sweep
    {
        size_t sim_number{};
        std::string matrix_filename{};
        size_t num_bit_nodes{}, num_check_nodes{};
        double exact_qber{};
        size_t frames{};
        size_t frame_iterations{}; // executed BP iterations summed over the frames
        double seconds{};          // wall time of the point (generation + transfers + decode, all GPUs)
    };
    struct sweep_report // throughput side-report of the last QKD_LDPC_batch_simulation (never written into the reference CSV)
    {
        double seconds_total{};
        double seconds_device{};
        double seconds_startup{}; // from entry until every GPU worker holds its context and the communicators exist (driver + context + NCCL initialisation)
        double seconds_comm_setup{}; // NCCL communicator set-up on the side thread (part of the start-up); 0 without a collective
        double seconds_reduce{};     // the all-reduce of the statistics itself, after the workers have stopped
        size_t frames{};
        size_t frame_iterations{};
        int gpus{};
        std::vector<point_report> points{};
    };
    const sweep_report &last_sweep_report();
    // Where QKD_LDPC_batch_simulation appends every finished point while it runs (`ldpc(...).partial.csv` in the reference's
    // format and `throughput(...).partial.csv`), so a 1 M-frame sweep holds nothing per trial and loses nothing on abort; the
    // files are removed when the sweep completes and the caller writes the final ones. Empty (default): no progress files.
    void set_progress_directory(const fs::path &directory);
    // Side file next to the reference-format CSV: per-point throughput, sifted-key rate, reconciliation efficiency
    // f = (1 - R) / h2(q) and leaked bits per frame (= M: plain syndrome coding). SURVEY.md 8f-3.
    void write_report(const sweep_report &report, fs::path directory);
    // Non-fatal findings about a loaded matrix (unsorted adjacency lists, duplicate edges); SURVEY.md 8f-2.
    std::vector<std::string> matrix_warnings(const H_matrix &matrix);
    // Seeded PEG construction of a column-weight-`dv` code, written as an alist file (host/peg.cpp).
    void generate_peg_alist(size_t n, size_t m, size_t dv, uint64_t seed, size_t bfs_limit, const fs::path &out_path);
    void release_device_state(); // frees cached device codes / contexts (also done at process exit)
}
