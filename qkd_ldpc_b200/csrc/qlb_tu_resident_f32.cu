#include "qlb_internal.hpp"
#include <algorithm>
using namespace qlb;
#include "qlb_resident_f32.cuh"

namespace
{
    // The specialised fp32 kernel (qlb_resident_f32.cuh): whole frame in shared memory, uniform bit weight.
    template <typename Rule, bool kReconcile, int kBW>
    int launch_resident(qlb_ctx *ctx, DecodeArgs &args)
    {
        auto kern = decode_resident_f32_kernel<Rule, kReconcile, kBW, kResidentThreads>;
        int kThreads = balanced_block_size(args.code, kResidentThreads, 0.55);
        if (const int t = args.block_threads / 32 * 32) // qlb_decode_params.block_threads
            if (t >= 32 && t <= kResidentThreads && 32 * t >= args.code.n && 32 * t >= args.code.m)
                kThreads = t;
        const size_t smem = resident_smem_bytes(args.code.n, args.code.m, args.code.slots, kBW);
        QLB_CUDA(allow_full_dynamic_smem(ctx, kern));
        long long grid = ctx->sm_count; // one resident CTA per SM
        if (grid > args.n_frames)
            grid = args.n_frames;
#ifdef QLB_BOUNDS_CHECK
        const uint32_t msg_bytes = 4u * (uint32_t)args.code.slots;
        QLB_CUDA(cudaMemcpyToSymbolAsync(g_bounds_msg_bytes, &msg_bytes, 4, 0, cudaMemcpyHostToDevice, ctx->stream));
#endif
        QLB_CUDA(cudaMemsetAsync(ctx->d_counters, 0, sizeof(unsigned long long), ctx->stream));
        args.queue = ctx->d_counters;
        args.iter_total = ctx->d_counters + 1;
        std::snprintf(ctx->last_decoder, sizeof ctx->last_decoder, "resident_f32%s bw=%d threads=%d",
                      std::is_same<Rule, RuleF32Fast>::value ? "fast" : "", kBW, kThreads);
        kern<<<(unsigned)grid, kThreads, smem, ctx->stream>>>(args);
        QLB_CUDA(cudaGetLastError());
        ++ctx->launches;
        return QLB_OK;
    }

    template <typename Rule, bool kReconcile>
    int launch_resident_bw(qlb_ctx *ctx, DecodeArgs &args)
    {
        switch (args.code.uniform_bit_w)
        {
        case 2: return launch_resident<Rule, kReconcile, 2>(ctx, args);
        case 3: return launch_resident<Rule, kReconcile, 3>(ctx, args);
        case 4: return launch_resident<Rule, kReconcile, 4>(ctx, args);
        default: return fail(QLB_ERR_UNSUPPORTED, "resident kernel: unsupported bit weight");
        }
    }

}
namespace qlb
{
    bool resident_f32_eligible(const qlb_ctx *ctx, const CodeDev &c)
    {
        return c.slots < 65535 && c.bit_slots16 && c.uniform_bit_w >= 2 && c.uniform_bit_w <= 4 && c.max_check_w <= kResidentMaxCW &&
               balanced_block_size(c, kResidentThreads, 0.55) > 0 && c.n % 32 == 0 &&
               resident_smem_bytes(c.n, c.m, c.slots, c.uniform_bit_w) + kResidentStaticSmem <= (size_t)ctx->smem_optin;
    }

    int launch_resident_f32(qlb_ctx *ctx, DecodeArgs &args, bool reconcile, bool fast)
    {
        if (fast)
            return reconcile ? launch_resident_bw<RuleF32Fast, true>(ctx, args) : launch_resident_bw<RuleF32Fast, false>(ctx, args);
        return reconcile ? launch_resident_bw<RuleF32Accurate, true>(ctx, args) : launch_resident_bw<RuleF32Accurate, false>(ctx, args);
    }
}
