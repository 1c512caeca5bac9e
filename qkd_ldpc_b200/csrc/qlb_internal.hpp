// Internal declarations shared by the translation units of libqkdldpc_b200.so (not part of the C-ABI).
// The library is split into TUs that compile in parallel: qlb_api.cu (C-ABI, code/context management, syndrome, key generator,
// trace) and one per decoder family, with its admission predicate and its launcher: qlb_tu_generic.cu, qlb_tu_resident_f32.cu,
// qlb_tu_resident_f64.cu, qlb_tu_stream.cu. route_decode, below, chooses the family of a batch. qlb_rate.cu turns rate-adapted
// batches into the sum-product mode every family takes.
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <map>
#include <string>
#include <tuple>
#include <type_traits>
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
    qlb::DevBuf rate_tab, rate_fill, rate_word, rate_key; // rate-adapted batches (qlb_rate.cu): class tables, fill, mother words, keys
    std::vector<double> host_logp;
    std::vector<uint32_t> host_pack_a, host_pack_b, host_pack_out;
    char last_decoder[128] = {}; // written by each decode launcher just before it launches (qlb_ctx_last_decoder)
};

namespace qlb
{
    struct CodeLayout;
    // qlb_api.cu: the host layout of a code, its device copy on a context, the parameter check every decode entry runs, and the
    // syndrome of packed device frames
    const CodeLayout &layout_of(const qlb_code *code);
    int get_device_code(qlb_ctx *ctx, const qlb_code *code, const CodeDev **out);
    int check_params(const qlb_decode_params *p);
    int launch_syndrome(qlb_ctx *ctx, const CodeDev &dev, long long n_frames, const uint32_t *d_bits, uint32_t *d_out);

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

    // the precision and its cheaper check rule (QLB_FLAG_F32_FAST_MATH / F64_FUSED_RATIO), or fp32 min-sum (QLB_FLAG_F32_MIN_SUM)
    enum class Rule { F64, F64Fused, F32, F32Fast, F32MinSum };
    enum class Family { ResidentF32, ResidentF64, Stream, Generic };
    struct Route // the decoder that takes a batch, and how it runs
    {
        Family family;
        Rule rule;
        bool reconcile; // reconcile mode (keys and log prior) or sum-product mode (LLRs and syndrome)
        Tier tier;      // generic kernel: storage tier
        int32_t stream_max_bundles, stream_no_repack, block_threads; // qlb_decode_params' execution knobs
    };

    // One TU per decoder family: admission predicate (fp64 resident: the code has group tables) and launcher.
    bool resident_f32_eligible(const qlb_ctx *ctx, const CodeDev &c);
    int launch_resident_f32(qlb_ctx *ctx, DecodeArgs &args, const Route &r);
    bool resident64_build_tables(const qlb_ctx *ctx, const CodeDev &c, const uint32_t *bit_slots, std::vector<uint32_t> &check_groups,
                                 std::vector<uint16_t> &bit_groups, uint32_t &smem_slots);
    int launch_resident_f64(qlb_ctx *ctx, DecodeArgs &args, const Route &r);
    bool stream_eligible(const CodeDev &c);
    int launch_stream(qlb_ctx *ctx, DecodeArgs &args, const Route &r);
    Tier generic_tier(const qlb_ctx *ctx, const CodeDev &c, bool fp32); // the fastest storage tier the code fits in
    int launch_generic(qlb_ctx *ctx, DecodeArgs &args, const Route &r);

    // The node arithmetic (qlb_kernels.cuh) of each rule in the generic kernel and the fp64 decoders.
    template <Rule kRule> using MathOf = std::tuple_element_t<(int)kRule, std::tuple<MathF64, MathF64Fused, MathF32, MathF32Fast, MathF32MinSum>>;

    // Calls f(rule, reconcile) with the route's rule and mode as std::integral_constant<Rule, ...> and std::bool_constant: template
    // arguments for a launcher. Only the listed rules, those the family implements (route_decode picks no other), are instantiated.
    template <Rule kRule, Rule... kMore, typename F>
    int with_rule(const Route &r, F &&f)
    {
        if constexpr (sizeof...(kMore) > 0)
            if (r.rule != kRule)
                return with_rule<kMore...>(r, f);
        if (r.reconcile)
            return f(std::integral_constant<Rule, kRule>{}, std::true_type{});
        return f(std::integral_constant<Rule, kRule>{}, std::false_type{});
    }

    // The launch of a persistent decoder: min(SMs x ctas_per_sm, frames) CTAs, each taking frames from the queue counter until
    // none is left. `scratch`: global scratch bytes per CTA (0: none). `decoder`: what qlb_ctx_last_decoder reports.
    template <typename Kernel>
    int launch_persistent(qlb_ctx *ctx, DecodeArgs &args, Kernel kern, int threads, size_t smem, int ctas_per_sm, size_t scratch,
                          const char *decoder)
    {
        QLB_CUDA(allow_full_dynamic_smem(ctx, kern));
        const long long grid = std::min<long long>((long long)ctx->sm_count * ctas_per_sm, args.n_frames);
        if (scratch)
        {
            QLB_CUDA(ctx->scratch.reserve((size_t)grid * scratch));
            args.scratch = static_cast<unsigned char *>(ctx->scratch.p);
            args.scratch_stride = scratch;
        }
#ifdef QLB_DEBUG_LAUNCH
        std::fprintf(stderr, "[qlb] %s: %d CTA/SM, grid=%lld, smem=%zu B, scratch=%zu B/CTA\n", decoder, ctas_per_sm, grid, smem, scratch);
#endif
        QLB_CUDA(cudaMemsetAsync(ctx->d_counters, 0, sizeof(unsigned long long), ctx->stream));
        std::snprintf(ctx->last_decoder, sizeof ctx->last_decoder, "%s", decoder);
        kern<<<(unsigned)grid, threads, smem, ctx->stream>>>(args);
        QLB_CUDA(cudaGetLastError());
        ++ctx->launches;
        return QLB_OK;
    }

    // The decoder of a batch of checked parameters: the order of the tests is the whole policy.
    inline int route_decode(const qlb_ctx *ctx, const CodeDev &c, const qlb_decode_params &p, bool reconcile, Route &out)
    {
        const bool fp32 = p.precision == QLB_PRECISION_F32;
        // test hook (QLB_FLAG_TEST_TIER_SHIFT; check_params admits 0 ... 3): -1 none, 0 ... 2 the generic kernel in that storage
        // tier or a slower one, 3 the streaming decoder
        const int hook = ((p.flags >> QLB_FLAG_TEST_TIER_SHIFT) & 0xF) - 1;
        Rule rule = fp32 ? Rule::F32 : Rule::F64;
        if (p.flags & (fp32 ? QLB_FLAG_F32_FAST_MATH : QLB_FLAG_F64_FUSED_RATIO)) // the precision's cheaper check rule
            rule = fp32 ? Rule::F32Fast : Rule::F64Fused;
        if (p.flags & QLB_FLAG_F32_MIN_SUM) // fp32 only, never with the fast rule (check_params)
            rule = Rule::F32MinSum;
        out = Route{Family::Generic, rule, reconcile, kTierGlobal, p.stream_max_bundles, p.stream_no_repack, p.block_threads};
        if (hook < 0 && (fp32 ? resident_f32_eligible(ctx, c) : c.r64_check_group_table != nullptr))
            out.family = fp32 ? Family::ResidentF32 : Family::ResidentF64;
        // frame-interleaved streaming through HBM: in fp32 every code the resident kernel rejects; in fp64 the block lengths whose
        // slot indices do not fit the generic kernel's shared-memory tiers
        else if ((hook == 3 || (hook < 0 && (fp32 || c.slots >= 65535))) && stream_eligible(c))
            out.family = Family::Stream;
        else if (hook == 3)
            return fail(QLB_ERR_UNSUPPORTED, "the streaming kernel does not handle this code / precision");
        else // tests may force a slower tier, never one that does not fit
            out.tier = (Tier)std::max<int>(generic_tier(ctx, c, fp32), hook);
        return QLB_OK;
    }

    // The decode of a batch: its route, the arguments every decoder reads, the launch.
    inline int launch_decode(qlb_ctx *ctx, const qlb_decode_params &p, bool reconcile, DecodeArgs &args)
    {
        Route r;
        if (const int rc = route_decode(ctx, args.code, p, reconcile, r))
            return rc;
        args.queue = ctx->d_counters;
        args.iter_total = ctx->d_counters + 1;
        args.max_it = p.max_iterations;
        args.enable_thr = p.enable_threshold;
        args.thr = p.threshold;
        args.cap_f32 = p.enable_threshold ? (float)p.threshold : INFINITY;
        args.ms_scale = p.min_sum_scale;
        switch (r.family)
        {
        case Family::ResidentF32: return launch_resident_f32(ctx, args, r);
        case Family::ResidentF64: return launch_resident_f64(ctx, args, r);
        case Family::Stream: return launch_stream(ctx, args, r);
        case Family::Generic: return launch_generic(ctx, args, r);
        }
        return fail(QLB_ERR_INVALID, "decode route: unknown decoder family");
    }
}
