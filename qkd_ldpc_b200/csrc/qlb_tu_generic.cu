#include "qlb_internal.hpp"
using namespace qlb;

namespace
{
    // The generic kernel (qlb_kernels.cuh): any code, its working set split between shared memory and scratch by storage tier.
    template <typename Math, int kTier, bool kReconcile, int kShapeW, int kThreads>
    int launch_one(qlb_ctx *ctx, DecodeArgs &args, const char *rule)
    {
        typedef typename Math::real Real;
        auto kern = decode_kernel<Math, kTier, kReconcile, kShapeW, kThreads>;
        const Carve cv = make_carve<Real, kTier>(args.code.n, args.code.m, args.code.slots, args.code.max_bit_w);
        QLB_CUDA(allow_full_dynamic_smem(ctx, kern)); // before the occupancy query: it holds the request to the kernel's opt-in
        int per_sm = 0;
        QLB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kThreads, cv.total_smem));
        if (per_sm < 1)
            return fail(QLB_ERR_UNSUPPORTED, "decode kernel does not fit on an SM for this code");
        char name[sizeof(qlb_ctx::last_decoder)];
        std::snprintf(name, sizeof name, "generic %s tier=%d shape=%d threads=%d", rule, kTier, kShapeW, kThreads);
        return launch_persistent(ctx, args, kern, kThreads, cv.total_smem, per_sm, cv.total_scratch, name);
    }

    template <typename Math, int kTier, bool kReconcile, int kThreads>
    int launch_shape(qlb_ctx *ctx, DecodeArgs &args, const char *rule)
    {
        const int cw = args.code.max_check_w, bw = args.code.max_bit_w;
        if constexpr (kTier != kTierGlobal) // register-tile variants exist for the shared-memory tiers only
        {
            if (bw <= 4 && cw <= 8)
                return launch_one<Math, kTier, kReconcile, 8, kThreads>(ctx, args, rule);
            if (bw <= 4 && cw <= 16)
                return launch_one<Math, kTier, kReconcile, 16, kThreads>(ctx, args, rule);
        }
        return launch_one<Math, kTier, kReconcile, 0, kThreads>(ctx, args, rule);
    }
}
namespace qlb
{
    Tier generic_tier(const qlb_ctx *ctx, const CodeDev &c, bool fp32)
    {
        if (c.slots >= 65535 || !c.bit_slots16) // the shared-memory tiers take 16-bit slot indices
            return kTierGlobal;
        // fp64 messages never fit a whole frame in shared memory; tier 1 keeps the messages in global scratch, of either type
        if (fp32 && make_carve<float, kTierSmemAll>(c.n, c.m, c.slots, c.max_bit_w).total_smem <= (size_t)ctx->smem_optin)
            return kTierSmemAll;
        if (make_carve<double, kTierSmemIdx>(c.n, c.m, c.slots, c.max_bit_w).total_smem <= (size_t)ctx->smem_optin)
            return kTierSmemIdx;
        return kTierGlobal;
    }

    int launch_generic(qlb_ctx *ctx, DecodeArgs &args, const Route &r)
    {
        static const char *const kRuleName[] = {"f64", "f64fused", "f32", "f32fast", "f32minsum"}; // indexed by Rule
        const char *name = kRuleName[(int)r.rule];
        return with_rule<Rule::F64, Rule::F64Fused, Rule::F32, Rule::F32Fast, Rule::F32MinSum>(r, [&](auto rule, auto reconcile) -> int
        {
            typedef MathOf<decltype(rule)::value> Math;
            constexpr bool kReconcile = decltype(reconcile)::value;
            if constexpr (sizeof(typename Math::real) == 4) // no fp64 route has tier 0 (generic_tier)
                if (r.tier == kTierSmemAll)
                    return launch_shape<Math, kTierSmemAll, kReconcile, 1024>(ctx, args, name);
            if (r.tier == kTierSmemIdx)
                return launch_shape<Math, kTierSmemIdx, kReconcile, 512>(ctx, args, name);
            return launch_shape<Math, kTierGlobal, kReconcile, 512>(ctx, args, name);
        });
    }
}
