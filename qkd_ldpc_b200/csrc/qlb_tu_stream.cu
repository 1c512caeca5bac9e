#include "qlb_internal.hpp"
#include <algorithm>
using namespace qlb;
#include "qlb_stream_split.cuh"

namespace
{
    // The streaming decoder (qlb_stream_split.cuh): one kernel per pass over all groups, in waves when device memory cannot
    // hold the message arrays of every group at once. Nothing here waits for the device.
    template <typename P, bool kReconcile, int kBW, int VEC>
    int launch_stream_split(qlb_ctx *ctx, DecodeArgs &args, size_t budget)
    {
        typedef typename P::real Real;
        const long long G = 32 * VEC, groups = (args.n_frames + G - 1) / G;
        // groups per bundle: 2 KB of contiguous memory per slot when there are enough groups (see qlb_stream_split.cuh)
        int B = VEC == P::kVecWide ? SplitTune<P>::kBundle : 1; // measured on B200, N = 100 000, fp32: B = 1 / 2 / 4 / 8 -> 0.589 / 0.668 / 0.789 / 0.783 of the copy bandwidth
        while (B > 1 && (groups < B || (unsigned long long)args.code.slots * B * G >= 0xFFFFFFFFull)) // row offsets are 32-bit
            B /= 2;
        if ((unsigned long long)args.code.slots * B * G >= 0xFFFFFFFFull)
            return fail(QLB_ERR_UNSUPPORTED, "streaming decoder: more than 2^32 message values per frame group");
        const size_t per_bundle = split_bundle_bytes(args.code.n, args.code.m, args.code.slots, VEC, B, (int)sizeof(Real));
        long long fit_bundles = (long long)(budget / per_bundle);
        if (args.stream_max_bundles > 0) // qlb_decode_params.stream_max_bundles: waves without filling the device memory
            fit_bundles = std::min<long long>(fit_bundles, args.stream_max_bundles);
        if (fit_bundles < 1)
            return fail(QLB_ERR_UNSUPPORTED, "streaming decoder: device memory cannot hold the messages of one bundle of frame groups");
        const long long bundles = (groups + B - 1) / B;
        const long long waves = (bundles + fit_bundles - 1) / fit_bundles;
        const long long bundles_per_wave = (bundles + waves - 1) / waves; // equal waves instead of full ones and a remainder
        const long long per_wave = bundles_per_wave * B;                  // groups
        if (args.n_frames >= 0xFFFFFFFFLL)
            return fail(QLB_ERR_UNSUPPORTED, "streaming decoder: more than 2^32 - 2 frames in one call");
        const size_t state_words = (size_t)per_wave * 12 + (size_t)bundles_per_wave + 16 + 3 * (size_t)per_wave * G;
        QLB_CUDA(ctx->scratch.reserve((size_t)bundles_per_wave * per_bundle + state_words * 4));
        SplitState st{};
        st.bundles = static_cast<unsigned char *>(ctx->scratch.p);
        st.bundle_stride = per_bundle;
        st.bundle = B;
#ifndef QLB_STREAM64_REPACK_PCT
#define QLB_STREAM64_REPACK_PCT 65
#endif
        // measured on B200, N = 100 000, QBER 0.085, fp32: 50 / 65 / 80 / 90 % -> 0.664 / 0.694 / 0.686 / 0.651 of peak; fp64: 0.442 / 0.465 / 0.472 / 0.368
        st.repack_pct = P::kLsbDecision ? 65 : QLB_STREAM64_REPACK_PCT;
        uint32_t *words = reinterpret_cast<uint32_t *>(st.bundles + (size_t)bundles_per_wave * per_bundle);
        st.act = words;
        st.bad = words + 4 * per_wave;
        st.succ = words + 8 * per_wave;
        st.list = words + 12 * per_wave;
        st.n_live = st.list + bundles_per_wave;
        st.repack = st.n_live + 4;
        st.fmap = st.n_live + 16;
        st.src_of = st.fmap + (size_t)per_wave * G;
        st.fmap_new = st.src_of + (size_t)per_wave * G;
        if (args.syndrome_out)
            QLB_CUDA(cudaMemsetAsync(args.syndrome_out, 0, (size_t)args.n_frames * args.code.words_m * 4, ctx->stream));
        args.queue = ctx->d_counters;
        args.iter_total = ctx->d_counters + 1;

        auto k_setup = stream_setup_kernel<Real, kReconcile, VEC>;
        auto k_init = stream_init_kernel<P, kReconcile, kBW, VEC>;
        auto k_check = stream_check_kernel<P, kReconcile, VEC>;
        auto k_update = stream_update_kernel<VEC>;
        auto k_bit = stream_bit_kernel<P, kReconcile, kBW, VEC>;
        auto k_final = stream_finalize_kernel<Real, kReconcile, VEC>;
        auto k_plan = stream_repack_plan_kernel<VEC>;
        auto k_mvmsg = stream_repack_msg_kernel<Real, VEC>;
        auto k_mvbits = stream_repack_bits_kernel<Real, VEC>;
        auto k_commit = stream_repack_commit_kernel<VEC>;
        // rounds after which a repack is attempted (decided on the device: live columns <= half of the streamed ones)
        const bool repack_on = !args.stream_no_repack && per_wave <= kMaxRepackGroups && per_wave >= 2;
        // attempts every 2 / 3 / 4 rounds measured 0.681 / 0.680 / 0.681 at the waterfall, but every second round costs the
        // early-converging QBERs 10 %; a declined attempt costs ~15 us
        auto repack_round = [](int it) { return it >= 4 && it % 4 == 2; };
        constexpr int kSplitCheckThreads = SplitTune<P>::kCheckThreads;
        int occ_check = 1, occ_bit = 1;
        QLB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_check, k_check, kSplitCheckThreads, 0));
        QLB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_bit, k_bit, kSplitBitThreads, 0));
        const unsigned grid_check = (unsigned)(ctx->sm_count * std::max(1, occ_check)), grid_bit = (unsigned)(ctx->sm_count * std::max(1, occ_bit));
#ifdef QLB_DEBUG_LAUNCH
            std::fprintf(stderr, "[qlb] stream split VEC=%d: %lld groups of %lld frames, bundles of %d, %lld wave(s) of <= %lld groups, %zu B per bundle; check grid %u (%d/SM), bit grid %u (%d/SM)\n",
                         VEC, groups, G, B, waves, per_wave, per_bundle, grid_check, occ_check, grid_bit, occ_bit);
#endif
        const char bw[2] = {kBW ? (char)('0' + kBW) : '\0', '\0'};
        std::snprintf(ctx->last_decoder, sizeof ctx->last_decoder, "stream_%s vec=%d bw=%s bundle=%d waves=%lld repack=%d",
                      sizeof(Real) == 4 ? "f32" : "f64", VEC, kBW ? bw : "any", B, waves, (int)repack_on);
        for (long long w = 0; w < waves; ++w)
        {
            st.group0 = w * per_wave;
            st.n_groups = (int)std::min<long long>(per_wave, groups - st.group0);
            if (st.n_groups <= 0)
                break;
            const unsigned grid_groups = (unsigned)std::min<long long>(st.n_groups, 2LL * ctx->sm_count);
            k_setup<<<grid_groups, kSplitSetupThreads, 0, ctx->stream>>>(args, st);
            k_init<<<grid_bit, kSplitBitThreads, 0, ctx->stream>>>(args, st);
            for (int it = 0;; ++it)
            {
                k_check<<<grid_check, kSplitCheckThreads, 0, ctx->stream>>>(args, st, it);
                k_update<<<1, 1024, 0, ctx->stream>>>(args, st, it);
                if (it == args.max_it)
                    break;
                if (repack_on && repack_round(it))
                {
                    k_plan<<<1, 1024, 0, ctx->stream>>>(st);
                    k_final<<<grid_groups, kSplitSetupThreads, 0, ctx->stream>>>(args, st, 1);
                    k_mvmsg<<<grid_bit, kRepackThreads, 0, ctx->stream>>>(args, st);
                    k_mvbits<<<grid_bit, kRepackThreads, 0, ctx->stream>>>(args, st);
                    k_commit<<<1, 1024, 0, ctx->stream>>>(st);
                    ctx->launches += 5;
                }
                k_bit<<<grid_bit, kSplitBitThreads, 0, ctx->stream>>>(args, st);
            }
            k_final<<<grid_groups, kSplitSetupThreads, 0, ctx->stream>>>(args, st, 0);
            QLB_CUDA(cudaGetLastError());
            ctx->launches += 3 + 3ULL * (unsigned)args.max_it + 2;
        }
        return QLB_OK;
    }

    template <typename P, bool kReconcile, int kBW>
    int launch_stream_vec(qlb_ctx *ctx, DecodeArgs &args)
    {
        size_t free_b = 0, total_b = 0;
        QLB_CUDA(cudaMemGetInfo(&free_b, &total_b));
        const size_t budget = (free_b + ctx->scratch.cap) / 20 * 17;
        // groups of 128 (fp32) / 64 (fp64) frames: 128-bit accesses; a batch of <= 32 frames takes 32-frame groups
        return args.n_frames > 32 ? launch_stream_split<P, kReconcile, kBW, P::kVecWide>(ctx, args, budget) : launch_stream_split<P, kReconcile, kBW, 1>(ctx, args, budget);
    }

    template <typename P, bool kReconcile>
    int launch_stream_bw(qlb_ctx *ctx, DecodeArgs &args)
    {
        switch (args.code.uniform_bit_w)
        {
#ifndef QLB_STREAM_LEAN // kernel-tuning builds (scripts/build_stream_variants.py) compile the bit weight of the benchmark codes only
        case 2: return launch_stream_vec<P, kReconcile, 2>(ctx, args);
        case 4: return launch_stream_vec<P, kReconcile, 4>(ctx, args);
#endif
        case 3: return launch_stream_vec<P, kReconcile, 3>(ctx, args);
        default: return launch_stream_vec<P, kReconcile, 0>(ctx, args); // irregular or heavier bits: the any-weight bit pass
        }
    }
}
namespace qlb
{
    // any bit weights (uniform 2 / 3 / 4 -- BASELINE.json's code family is CW = 3 -- through register-tiled instantiations of the bit
    // pass, everything else through the any-weight form); check weights up to 16
    bool stream_eligible(const CodeDev &c)
    {
        return c.max_bit_w >= 1 && c.max_check_w <= kResidentMaxCW && c.m <= c.n && c.col_of_slot32 != nullptr;
    }
    int launch_stream_f32(qlb_ctx *ctx, DecodeArgs &args, bool reconcile, bool fast)
    {
        if (fast)
            return reconcile ? launch_stream_bw<StreamF32<RuleF32Fast>, true>(ctx, args) : launch_stream_bw<StreamF32<RuleF32Fast>, false>(ctx, args);
        return reconcile ? launch_stream_bw<StreamF32<RuleF32Accurate>, true>(ctx, args) : launch_stream_bw<StreamF32<RuleF32Accurate>, false>(ctx, args);
    }
    int launch_stream_f64(qlb_ctx *ctx, DecodeArgs &args, bool reconcile, bool fused)
    {
        if (fused)
            return reconcile ? launch_stream_bw<StreamF64<MathF64Fused>, true>(ctx, args) : launch_stream_bw<StreamF64<MathF64Fused>, false>(ctx, args);
        return reconcile ? launch_stream_bw<StreamF64<MathF64>, true>(ctx, args) : launch_stream_bw<StreamF64<MathF64>, false>(ctx, args);
    }
}
