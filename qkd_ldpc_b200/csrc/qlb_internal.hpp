// Internal declarations shared by the translation units of libqkdldpc_b200.so (not part of the C-ABI).
// The library is split into one TU per kernel family so that they compile in parallel:
//   qlb_api.cu            C-ABI, code/context management, generic decode_kernel, syndrome, key generator
//   qlb_tu_resident_f32.cu / qlb_tu_stream_f32.cu / qlb_tu_resident_f64.cu   the specialised decoders + their launchers
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <map>
#include <string>
#include <vector>

#include "../../include/qkd_ldpc_b200.h"
#include "qlb_kernels.cuh"

namespace qlb
{
    int fail(int code, const std::string &msg);
    int cuda_fail(cudaError_t e, const char *what);
}
#define QLB_CUDA(call)                                   \
    do                                                   \
    {                                                    \
        cudaError_t e__ = (call);                        \
        if (e__ != cudaSuccess)                          \
            return qlb::cuda_fail(e__, #call);           \
    } while (0)

namespace qlb
{
    struct DeviceCode
    {
        CodeDev dev{};
        std::vector<void *> allocs;
    };

    // grow-only device buffer
    struct DevBuf
    {
        void *p = nullptr;
        size_t cap = 0;
        cudaError_t reserve(size_t bytes)
        {
            if (bytes <= cap)
                return cudaSuccess;
            if (p)
                cudaFree(p);
            p = nullptr;
            cap = 0;
            cudaError_t e = cudaMalloc(&p, bytes);
            if (e == cudaSuccess)
                cap = bytes;
            return e;
        }
        void release()
        {
            if (p)
                cudaFree(p);
            p = nullptr;
            cap = 0;
        }
    };
}

struct qlb_ctx
{
    int device = 0;
    int sm_count = 0;
    int smem_optin = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev_start = nullptr, ev_stop = nullptr;
    unsigned long long *d_counters = nullptr; // [0] frame queue, [1] executed iterations
    uint64_t launches = 0;
    std::map<uint64_t, qlb::DeviceCode> codes;
    qlb::DevBuf scratch, in_a, in_b, in_q, in_llr, in_syn, out_it, out_res, out_dec, out_syn, gen_perm, gen_seeds;
    std::vector<double> host_logp;
    std::vector<uint32_t> host_pack_a, host_pack_b, host_pack_out;
    char last_decoder[128] = {}; // written by each decode launcher just before it launches (qlb_ctx_last_decoder)
};

namespace qlb
{
    // Opt a kernel in to the device's whole per-block shared memory. ALWAYS the same value for a given kernel -- the attribute belongs
    // to the function, not to the launch, and contexts are driven from several host threads at once: setting it to what the current
    // launch needs lets another thread's smaller request land between this thread's set and its launch ("invalid argument").
    template <typename Kernel>
    inline cudaError_t allow_full_dynamic_smem(const qlb_ctx *ctx, Kernel kern)
    {
        cudaFuncAttributes fa;
        cudaError_t e = cudaFuncGetAttributes(&fa, kern);
        if (e != cudaSuccess)
            return e;
        return cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, ctx->smem_optin - (int)fa.sharedSizeBytes);
    }

    // Block size (multiple of 32, in [max/2, max]) for the thread-per-node kernels. Every thread walks the bits with stride T and each
    // weight segment of the sorted checks with stride T, and the block waits for the slowest thread, so T is chosen to keep the
    // last round of each walk as full as possible (`check_share`: the check walk's share of an iteration); among equally balanced
    // sizes the smaller block measured slightly faster (B200, N=10240: 768 > 896 > 1024 threads by 2 %). Both walks must stay within the 32 per-thread rounds the kernels park bits for.
    // `min_threads`: the fp64 kernel is latency-bound (dependent DFMA chains, L2 index loads) and wants warps more than balance:
    // measured on B200, N=10240, fused rule: 384 / 512 / 640 / 768 threads = 3.08 / 3.46 / 3.61 / 3.87 M frame-iterations/s
    // (`size_bias` > 0: among equally balanced sizes the larger block).
    inline int balanced_block_size(const CodeDev &c, int max_threads, double check_share, int min_threads = 0, double size_bias = -0.02)
    {
        int best = 0;
        double best_score = -1.;
        if (min_threads <= 0)
            min_threads = max_threads / 2;
        for (int t = max_threads; t >= min_threads && t >= 32; t -= 32)
        {
            long long check_rounds = 0;
            for (int w = c.max_check_w; w >= 0; --w)
            {
                const long long lo = (w < c.max_check_w) ? c.cnt[w] : 0, hi = (w > 0) ? c.cnt[w - 1] : c.m;
                check_rounds += (hi - lo + t - 1) / t;
            }
            const long long bit_rounds = (c.n + t - 1) / t;
            if (check_rounds > 32 || bit_rounds > 32)
                break;
            const double ec = (double)c.m / t / (double)check_rounds, eb = (double)c.n / t / (double)bit_rounds;
            const double score = (check_share * ec + (1. - check_share) * eb) * (1. + size_bias * t / max_threads);
            if (score > best_score + 1e-12)
            {
                best_score = score;
                best = t;
            }
        }
        return best; // 0: no admissible block size
    }

    // launchers of the specialised decoders (each in its own TU); `fast`: the SFU check rule
    bool resident_f32_eligible(const qlb_ctx *ctx, const CodeDev &c);
    int launch_resident_f32(qlb_ctx *ctx, DecodeArgs &args, bool reconcile, bool fast);
    bool stream_eligible(const CodeDev &c);
    int launch_stream_f32(qlb_ctx *ctx, DecodeArgs &args, bool reconcile, bool fast);
    int launch_stream_f64(qlb_ctx *ctx, DecodeArgs &args, bool reconcile, bool fused); // `fused`: the fused-ratio check rule
    bool resident_f64_eligible(const qlb_ctx *ctx, const CodeDev &c);
    bool resident64_build_tables(const qlb_ctx *ctx, const CodeDev &c, const uint32_t *bit_slots, std::vector<uint32_t> &check_groups,
                                 std::vector<uint16_t> &bit_groups, uint32_t &smem_slots);
    int launch_resident_f64(qlb_ctx *ctx, DecodeArgs &args, bool reconcile, bool fused);
}
