#include "qlb_internal.hpp"
using namespace qlb;
#include "qlb_resident_f32.cuh"

namespace
{
    // Block size (multiple of 32, in [max/2, max]). Every thread walks the bits with stride T and each weight segment of the sorted
    // checks with stride T, and the block waits for the slowest thread, so T is chosen to keep the last round of each walk as full
    // as possible (`check_share`: the check walk's share of an iteration); among equally balanced sizes the smaller block measured
    // slightly faster (B200, N=10240: 768 > 896 > 1024 threads by 2 %). Both walks must stay within the 32 per-thread rounds the kernel parks bits for.
    int balanced_block_size(const CodeDev &c, int max_threads, double check_share)
    {
        int best = 0;
        double best_score = -1.;
        for (int t = max_threads; t >= max_threads / 2 && t >= 32; t -= 32)
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
            const double score = (check_share * ec + (1. - check_share) * eb) * (1. - 0.02 * t / max_threads);
            if (score > best_score + 1e-12)
            {
                best_score = score;
                best = t;
            }
        }
        return best; // 0: no admissible block size
    }

    // The specialised fp32 kernel (qlb_resident_f32.cuh): whole frame in shared memory, uniform bit weight.
    template <typename CheckRule, bool kReconcile, int kBW>
    int launch_resident(qlb_ctx *ctx, DecodeArgs &args, int block_threads)
    {
        auto kern = decode_resident_f32_kernel<CheckRule, kReconcile, kBW, kResidentThreads>;
        int kThreads = balanced_block_size(args.code, kResidentThreads, 0.55);
        if (const int t = block_threads / 32 * 32) // qlb_decode_params.block_threads
            if (t >= 32 && t <= kResidentThreads && 32 * t >= args.code.n && 32 * t >= args.code.m)
                kThreads = t;
        const size_t smem = resident_smem_bytes(args.code.n, args.code.m, args.code.slots, kBW);
#ifdef QLB_BOUNDS_CHECK
        const uint32_t msg_bytes = 4u * (uint32_t)args.code.slots;
        QLB_CUDA(cudaMemcpyToSymbolAsync(g_bounds_msg_bytes, &msg_bytes, 4, 0, cudaMemcpyHostToDevice, ctx->stream));
#endif
        char name[sizeof(qlb_ctx::last_decoder)];
        const char *rule = std::is_same<CheckRule, RuleF32Fast>::value ? "fast" : std::is_same<CheckRule, RuleF32MinSum>::value ? "minsum" : "";
        std::snprintf(name, sizeof name, "resident_f32%s bw=%d threads=%d", rule, kBW, kThreads);
        return launch_persistent(ctx, args, kern, kThreads, smem, 1, 0, name); // one resident CTA per SM
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

    int launch_resident_f32(qlb_ctx *ctx, DecodeArgs &args, const Route &r)
    {
        return with_rule<Rule::F32, Rule::F32Fast, Rule::F32MinSum>(r, [&](auto rule, auto reconcile) -> int
        {
            typedef std::tuple_element_t<(int)decltype(rule)::value - (int)Rule::F32, std::tuple<RuleF32Accurate, RuleF32Fast, RuleF32MinSum>> CheckRule;
            constexpr bool kReconcile = decltype(reconcile)::value;
            switch (args.code.uniform_bit_w)
            {
            case 2: return launch_resident<CheckRule, kReconcile, 2>(ctx, args, r.block_threads);
            case 3: return launch_resident<CheckRule, kReconcile, 3>(ctx, args, r.block_threads);
            case 4: return launch_resident<CheckRule, kReconcile, 4>(ctx, args, r.block_threads);
            default: return fail(QLB_ERR_UNSUPPORTED, "resident kernel: unsupported bit weight");
            }
        });
    }
}
