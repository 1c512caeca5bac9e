/*
 * qkd_ldpc_b200.h -- C-ABI of libqkdldpc_b200.so
 *
 * B200-native (sm_100a) replacement for the hot path of ColdCloudd/QKD_LDPC: syndrome-based LDPC
 * information reconciliation by flooding sum-product belief propagation. Plain pointers and sizes
 * only; no C++ or torch types cross this boundary. There is NO CPU fallback behind these entry
 * points: every compute call fails with QLB_ERR_CUDA when no sm_100-class device is usable.
 *
 * Each entry point names the reference interface it replaces (paths relative to the reference
 * repository root). The host-side C++ mirror of the reference API (qkd_ldpc_b200/host/) and the
 * Python binding (qkd_ldpc_b200/capi.py) are thin callers of exactly these functions.
 *
 * Conventions (same as the reference unless noted):
 *   - a key / syndrome bit is 0 or 1; "unpacked" arrays hold one 32-bit int per bit
 *     (src/array_and_matrix_operations.hpp:39-40); "packed" arrays hold 32 bits per uint32_t word,
 *     bit i of a frame in word i/32 at bit position i%32, frames padded to whole words
 *     (row stride qlb_code_words_n() / qlb_code_words_m() words); the padding bits of a packed input
 *     are ignored, and those of a packed output are zero;
 *   - LLR sign: positive means bit 0 (src/qkd_ldpc_algorithm.cpp:259-266,401-405);
 *   - node indices are 0-based (src/array_and_matrix_operations.cpp:255,276);
 *   - all host buffers are owned by the caller; the library owns device scratch inside a context.
 *
 * Thread safety: a qlb_code is immutable after creation and may be shared; a qlb_ctx must be used
 * by one host thread at a time (one context per GPU per thread, as the reference uses one scratch
 * set per pool worker, src/simulation.cpp:230,244-250).
 */
#ifndef QKD_LDPC_B200_H
#define QKD_LDPC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define QLB_VERSION 200 /* 0.2.0: qlb_decode_params grew execution knobs (was 24 bytes, now 40) */

/* status codes (0 = ok); qlb_last_error() gives the message of the calling thread's last failure */
enum {
    QLB_OK = 0,
    QLB_ERR_INVALID = 1,     /* bad argument / inconsistent matrix                                  */
    QLB_ERR_CUDA = 2,        /* CUDA runtime failure or no usable device                            */
    QLB_ERR_UNSUPPORTED = 3, /* valid input the kernels do not handle (see message)                 */
    QLB_ERR_KEY_TOO_SMALL = 4, /* floor(N*QBER) == 0: the reference throws here (src/simulation.cpp:170-175) */
    QLB_ERR_NCCL = 5
};

/* message arithmetic */
enum {
    QLB_PRECISION_F64 = 64, /* the reference's arithmetic and operation order (tanh, divide, 2*atanh) */
    QLB_PRECISION_F32 = 32  /* single precision, leave-one-out products (no reference counterpart)    */
};

/* qlb_decode_params.flags */
enum {
    QLB_FLAG_F32_FAST_MATH = 1, /* fp32 only: exp-domain check rule on MUFU ex2/lg2/rcp instead of tanhf/atanhf */
    /* fp64 only: the check rule src/qkd_ldpc_algorithm.cpp:220-243 evaluated as ln((S - e D) / (D - e S)) -- one exp, one
     * division, one log per edge instead of tanh, divide, atanh. Same function, different rounding near saturation; honoured
     * by the SM-resident fp64 kernel and by the generic kernel (checks wider than its unrolled shapes keep the literal order).
     * Per-frame outcomes validated against the reference in profiles/parity_r01.md and on the exhaustive small-code fixtures. */
    QLB_FLAG_F64_FUSED_RATIO = 2,
    /* test hook, bits 8..11 = 1 + storage tier (0 shared memory, 1 L2 scratch for messages, 2 all global): run the generic
     * kernel in that tier instead of the fastest eligible one; ignored when the tier does not fit */
    QLB_FLAG_TEST_TIER_SHIFT = 8
};

typedef struct qlb_code qlb_code; /* a parity-check matrix prepared for the device (replaces H_matrix on the device side) */
typedef struct qlb_ctx qlb_ctx;   /* one GPU: stream, scratch, device copies of the codes it has seen */

/* Mirrors what the reference reads from the global CFG inside the hot path
 * (src/qkd_ldpc_algorithm.cpp:246,313,424-425; src/config.hpp:40-58). */
typedef struct qlb_decode_params {
    int32_t precision;        /* QLB_PRECISION_F64 | QLB_PRECISION_F32                              */
    int32_t max_iterations;   /* CFG.SUM_PRODUCT_MAX_ITERATIONS, >= 1                               */
    int32_t enable_threshold; /* CFG.ENABLE_SUM_PRODUCT_MSG_LLR_THRESHOLD                           */
    int32_t flags;            /* QLB_FLAG_*                                                        */
    double threshold;         /* CFG.SUM_PRODUCT_MSG_LLR_THRESHOLD, > 0 when enabled                */
    /* Execution knobs with no effect on results (0 = library default). They replace what used to be environment
     * variables: a drop-in library is steered through its arguments only. */
    int32_t stream_max_bundles; /* streaming decoder: at most this many 4-group bundles per wave (default: what device memory holds) */
    int32_t stream_no_repack;   /* streaming decoder: 1 = no on-device compaction of the live frames                  */
    int32_t block_threads;      /* SM-resident decoders: threads per CTA (multiple of 32; ignored when inadmissible)   */
    int32_t reserved;           /* must be 0                                                                           */
} qlb_decode_params;

/* Per-frame result of a decode; mirrors SP_result / LDPC_result (src/qkd_ldpc_algorithm.hpp:14-24). */
enum { QLB_RES_SYNDROMES_MATCH = 1, QLB_RES_KEYS_MATCH = 2 };

int qlb_version(void);
const char *qlb_last_error(void);

/* Number of visible CUDA devices (0 when none); never fails. */
int qlb_device_count(void);

/* ---- code handle ------------------------------------------------------------------------------
 * Replaces the device-facing role of `struct H_matrix` (src/array_and_matrix_operations.hpp:16-27).
 * Input is the matrix flattened from that struct, both adjacency halves in stored order:
 *   check_nodes[j][k] = col_idx[row_ptr[j] + k],  check_nodes_weight[j] = row_ptr[j+1] - row_ptr[j]
 *   bit_nodes[i][k]   = row_idx[col_ptr[i] + k],  bit_nodes_weight[i]   = col_ptr[i+1] - col_ptr[i]
 * The reference routes messages positionally (arrival counters, src/qkd_ldpc_algorithm.cpp:228-243,
 * 300-311); creation replays those counters to fix the per-node operation order, and rejects
 * (QLB_ERR_INVALID) matrices whose two halves do not describe the same edges in the same order
 * -- the inputs on which the reference itself would misroute or overrun its rows.
 */
int qlb_code_create(int32_t n_bits, int32_t n_checks, const int32_t *row_ptr, const int32_t *col_idx,
                    const int32_t *col_ptr, const int32_t *row_idx, qlb_code **code_out);
void qlb_code_destroy(qlb_code *code);
int32_t qlb_code_n(const qlb_code *code);       /* bit nodes   */
int32_t qlb_code_m(const qlb_code *code);       /* check nodes */
int32_t qlb_code_edges(const qlb_code *code);   /* edges       */
int32_t qlb_code_words_n(const qlb_code *code); /* uint32 words per packed key      = ceil(n/32) */
int32_t qlb_code_words_m(const qlb_code *code); /* uint32 words per packed syndrome = ceil(m/32) */

/* Test/inspection hook: copies the device layout tables into caller buffers (any may be NULL).
 *   slot_of_edge[e]  physical message slot (< qlb_code_slots()) of check-side edge e (CSR position)
 *   bit_slots[a*n+i] physical slot of the a-th message of bit i in the reference's summation order
 *                    (0xFFFFFFFF when a >= weight of bit i); a < qlb_code_max_bit_weight()
 *   check_order[p]   original check index handled at sorted position p
 */
int32_t qlb_code_max_bit_weight(const qlb_code *code);
int32_t qlb_code_max_check_weight(const qlb_code *code);
int32_t qlb_code_slots(const qlb_code *code);
int qlb_code_layout(const qlb_code *code, uint32_t *slot_of_edge, uint32_t *bit_slots, uint32_t *check_order);
/* Mean shared-memory wavefronts per warp-wide message gather of the bit pass (1.0 = conflict free): for the checks in
 * plain sorted order, and after the bank-aware placement the layout actually uses. */
int qlb_code_gather_wavefronts(const qlb_code *code, double *naive_out, double *placed_out);

/* ---- context ---------------------------------------------------------------------------------- */
int qlb_ctx_create(int device, qlb_ctx **ctx_out);
void qlb_ctx_destroy(qlb_ctx *ctx);
int qlb_ctx_device(const qlb_ctx *ctx);
int qlb_ctx_sm_count(const qlb_ctx *ctx);
/* The context's CUDA stream (a cudaStream_t) for callers that time or order work with their own events. */
void *qlb_ctx_stream(const qlb_ctx *ctx);
/* Which decoder the context's last decode launched, written by the launcher itself (empty before the first decode):
 *   "generic f64|f64fused|f32|f32fast tier=T shape=S threads=K"       the generic kernel (storage tier, unrolled check shape)
 *   "resident_f64[fused] bw=B threads=K smem_slots=X/S"             the SM-resident fp64 kernel (X of S message slots in shared memory)
 *   "resident_f32[fast] bw=B threads=K"                             the SM-resident fp32 kernel
 *   "stream_f32|f64 vec=V bw=B|any bundle=B waves=W repack=0|1"     the streaming decoder
 * The string is owned by the context and valid until its next decode. */
const char *qlb_ctx_last_decoder(const qlb_ctx *ctx);
int qlb_ctx_synchronize(qlb_ctx *ctx);
/* Decode-kernel launches and executed frame-iterations since the context was created / last reset. */
int qlb_ctx_counters(qlb_ctx *ctx, uint64_t *kernel_launches, uint64_t *frame_iterations, int reset);
/* CUDA-event stopwatch on the context's stream: start, enqueue work, stop -> elapsed milliseconds. */
int qlb_ctx_timer_start(qlb_ctx *ctx);
int qlb_ctx_timer_stop(qlb_ctx *ctx, float *elapsed_ms_out);

/* ---- syndrome ---------------------------------------------------------------------------------
 * Replaces calculate_syndrome_regular / calculate_syndrome_irregular
 * (src/array_and_matrix_operations.cpp:463-473 / 476-486) for a batch of frames:
 *   syndrome[f][j] = XOR_k bits[f][check_nodes[j][k]].
 * Host buffers; bits [n_frames][n], syndrome_out [n_frames][m] (unpacked) or word-padded (packed).
 */
int qlb_syndrome_batch(qlb_ctx *ctx, const qlb_code *code, int64_t n_frames, const int32_t *bits, int32_t *syndrome_out);
int qlb_syndrome_batch_packed(qlb_ctx *ctx, const qlb_code *code, int64_t n_frames, const uint32_t *bits_packed,
                              uint32_t *syndrome_packed_out);

/* ---- sum-product decode ------------------------------------------------------------------------
 * Replaces sum_product_decoding_regular / _irregular (src/qkd_ldpc_algorithm.cpp:3-173 / 175-345)
 * for a batch: a-priori LLRs llr[f][n] (double, as in the reference signature), target syndromes
 * syndrome[f][m] (unpacked). Outputs per frame: bits_out[f][n] (last hard decision, unpacked; may be
 * NULL), iterations_out[f] (SP_result.iterations_num), result_out[f] (QLB_RES_SYNDROMES_MATCH bit).
 */
int qlb_sum_product_batch(qlb_ctx *ctx, const qlb_code *code, const qlb_decode_params *params, int64_t n_frames,
                          const double *llr, const int32_t *syndrome, int32_t *bits_out, uint32_t *iterations_out,
                          uint8_t *result_out);

/* Trace form of ONE fp64 decode: what the reference prints under CFG.TRACE_SUM_PRODUCT / TRACE_SUM_PRODUCT_LLR
 * (src/qkd_ldpc_algorithm.cpp:214-327, 246-255 "E", 268-276 "L"/"z", 279-283 "s", 317-327 "M"), copied out per iteration
 * for the first `capacity` iterations (clamped to max_iterations). llr[n], syndrome[m] as in qlb_sum_product_batch.
 *   e_out[t][E]  check_to_bit_msg after the clamp, rows = bits in order, row i = its weight(i) slots in arrival order
 *   l_out[t][n]  total_bit_llr;  z_out[t][n] hard decision;  s_out[t][m] its syndrome
 *   m_out[t][E]  bit_to_check_msg after the clamp, rows = checks in order (not produced for the converging iteration)
 * E = number of edges; any of e/l/z/s/m_out and bits_out[n] may be NULL. precision must be QLB_PRECISION_F64. The
 * decision, iteration count and result equal qlb_sum_product_batch's on the same frame. */
int qlb_sum_product_trace(qlb_ctx *ctx, const qlb_code *code, const qlb_decode_params *params, const double *llr,
                          const int32_t *syndrome, int32_t capacity, double *e_out, double *l_out, int32_t *z_out,
                          int32_t *s_out, double *m_out, int32_t *bits_out, uint32_t *iterations_out, uint8_t *result_out);

/* ---- reconciliation ----------------------------------------------------------------------------
 * Replaces QKD_LDPC_regular / QKD_LDPC_irregular (src/qkd_ldpc_algorithm.cpp:347-396 / 398-447) for a
 * batch: per frame, prior +-ln((1-q)/q) from Bob's bits, Alice's syndrome, decode, key compare --
 * fused in one kernel. qber[f] is the frame's exact error ratio (src/simulation.cpp:169,183), must be
 * in (0,1). Outputs: iterations_out[f], result_out[f] (QLB_RES_* bits), optional decoded key
 * (which the reference computes and discards, :444) and optional Alice syndrome.
 */
int qlb_reconcile_batch(qlb_ctx *ctx, const qlb_code *code, const qlb_decode_params *params, int64_t n_frames,
                        const int32_t *alice, const int32_t *bob, const double *qber, uint32_t *iterations_out,
                        uint8_t *result_out, int32_t *decoded_out, int32_t *syndrome_out);
int qlb_reconcile_batch_packed(qlb_ctx *ctx, const qlb_code *code, const qlb_decode_params *params, int64_t n_frames,
                               const uint32_t *alice_packed, const uint32_t *bob_packed, const double *qber,
                               uint32_t *iterations_out, uint8_t *result_out, uint32_t *decoded_packed_out,
                               uint32_t *syndrome_packed_out);

/* Same operation on DEVICE-resident packed buffers (all pointers are device pointers on the context's
 * GPU; log_prior[f] = ln((1-q)/q) as a double). Enqueued on the context's stream, returns without
 * synchronizing. This is the entry the frame-batch scheduler and bench.py's device-resident leg use. */
int qlb_reconcile_device(qlb_ctx *ctx, const qlb_code *code, const qlb_decode_params *params, int64_t n_frames,
                         const uint32_t *d_alice_packed, const uint32_t *d_bob_packed, const double *d_log_prior,
                         uint32_t *d_iterations_out, uint8_t *d_result_out, uint32_t *d_decoded_packed_out,
                         uint32_t *d_syndrome_packed_out);

/* ---- key / error generation on the device ---------------------------------------------------------
 * Replaces, bit for bit, the inputs run_trial builds per trial (src/simulation.cpp:163-169): Alice's key from
 * generate_random_bit_array and Bob's from introduce_errors (src/array_and_matrix_operations.cpp:424-460), drawn from
 * XoshiroCpp::Xoshiro256PlusPlus(seeds[f] + seed_offset) with libstdc++ 13.3's uniform_int_distribution / std::shuffle
 * semantics. `qber` is the requested error probability; exactly floor(n_bits * qber) positions are flipped and
 * *exact_qber_out (optional) receives that count / n_bits. Fails with QLB_ERR_KEY_TOO_SMALL when it is zero
 * (the reference throws "Key size ... is too small for QBER.", src/simulation.cpp:170-175).
 * Keys come back packed; the _device form writes device buffers on the context's stream and does not synchronize.
 */
int qlb_generate_batch_packed(qlb_ctx *ctx, int32_t n_bits, int64_t n_frames, const uint64_t *seeds, uint64_t seed_offset, double qber,
                              uint32_t *alice_packed_out, uint32_t *bob_packed_out, double *exact_qber_out);
int qlb_generate_device(qlb_ctx *ctx, int32_t n_bits, int64_t n_frames, const uint64_t *d_seeds, uint64_t seed_offset, double qber,
                        uint32_t *d_alice_packed_out, uint32_t *d_bob_packed_out, double *exact_qber_out);
/* run_trial for a batch (src/simulation.cpp:161-189): keys generated on the device from the trial seeds, then reconciled;
 * only 8 bytes per frame go up and 5 come back. Host buffers. */
int qlb_run_trials(qlb_ctx *ctx, const qlb_code *code, const qlb_decode_params *params, int64_t n_frames, const uint64_t *seeds,
                   uint64_t seed_offset, double qber, uint32_t *iterations_out, uint8_t *result_out, double *exact_qber_out);

/* Test probe (no reference counterpart): the fp64 building blocks of the check rule, element-wise over host arrays, so that
 * their accuracy against the host libm is a test and not a claim. op 0: a / b (the rule's own division), 1: e^a for a in
 * [-64, 0], 2: ln(a / b) for 0 < b <= a, 3: tanh(a / 2), 4: 2 atanh(a) (b != 0: IEEE infinities at |a| = 1), 5: e^-|a| (the table-driven
 * form the check rules use). b may be NULL for the unary ops. */
int qlb_test_f64_math(qlb_ctx *ctx, int op, int64_t n, const double *a, const double *b, double *out);

/* ---- sweep statistics ---------------------------------------------------------------------------
 * The one collective of a sweep: element-wise SUM over the GPUs of one process of per-GPU integer statistics
 * (histogram of iterations_num over successful frames + counters; the quantities the reference accumulates serially at
 * src/simulation.cpp:252-312). vectors[g] is a HOST array of `count` uint64 owned by the caller for ctxs[g]; on return
 * every vectors[g] holds the sum. One ncclAllReduce per GPU inside a group call over NVLink (libnccl.so.2 is loaded on
 * first use; QLB_ERR_NCCL when it is missing or fails). With n_ctx == 1 the call is a device round trip through NCCL.
 * (Across processes -- one rank per GPU under torchrun -- the same reduction is done with torch.distributed/NCCL by
 * qkd_ldpc_b200/sweep.py.)
 */
int qlb_stats_allreduce(qlb_ctx *const *ctxs, int n_ctx, uint64_t *const *vectors, size_t count);
/* Creates (and keeps) the NCCL communicators qlb_stats_allreduce will use for contexts on these devices (in this order), and
 * nothing else: no collective runs. Communicator set-up takes seconds on an 8-GPU box; a sweep scheduler calls this from a side
 * thread as it starts, so that the set-up runs beside the CUDA start-up of the devices and the all-reduce at the end of the
 * sweep finds the communicators ready. Optional: qlb_stats_allreduce creates them itself when they are missing. */
int qlb_stats_comm_prepare(const int32_t *devices, int n_devices);

#ifdef __cplusplus
}
#endif
#endif /* QKD_LDPC_B200_H */
